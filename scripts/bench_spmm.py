"""Full-graph SpMM micro-benchmark (SURVEY.md section 8 f1: eval.py:47-70 aggregates over the WHOLE graph):
Y = A_hat X on the products-shaped graph with the default aggregation (form chosen by shape) and with the register-staged
kernels (grapes_agg_variant 1), bitwise compared and timed with CUDA events.  Also the frontier-shaped gather (n rows,
~1 source each)."""
import os, sys, json
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import build_workload
from grapes_b200._lib import lib, ptr
from grapes_b200.graph import DeviceGraph


def run(L, ctx, X, F, nodes, n, in_off, in_src, dinv, variant, reps=5, hi_lo=False, ldo=None, do_flush=True):
    ldo = ldo or F
    dev = X.device
    cnt = torch.tensor([n], dtype=torch.int32, device=dev)
    out = torch.zeros(n, ldo, dtype=torch.float32, device=dev)
    out_lo = torch.zeros(n, ldo, dtype=torch.float32, device=dev) if hi_lo else None
    L.cdll.grapes_agg_variant(variant)
    st = torch.cuda.current_stream().cuda_stream
    def call():
        L.grapes_aggregate(ctx, ptr(X), F, F, ptr(nodes), cnt.data_ptr(), n, ptr(in_off), ptr(in_src), ptr(dinv), None, 0,
                           None, 0, None if hi_lo else ptr(out), ldo, ptr(out) if hi_lo else None, ptr(out_lo), -1, st)
    call(); torch.cuda.synchronize()
    flush = torch.zeros(256 << 20, dtype=torch.uint8, device=dev)
    ts = []
    for _ in range(reps):
        if do_flush:
            flush.sum()                                 # L2 flush between timed launches: READ 256 MB (clean lines; a memset
                                                        # leaves 126 MB of dirty lines whose write-back lands in the timed kernel)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); call(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return out, ts[len(ts) // 2]


def main():
    which = sys.argv[1] if len(sys.argv) > 1 else "products"
    variants = (0, 1)
    dev = torch.device("cuda", 0)
    cfg, indptr, indices, x, y, train_idx = build_workload(which, 0, dev)
    N, F = cfg["N"], cfg["F"]
    g = DeviceGraph(indptr, indices, N)
    L = lib()
    res = {}
    # ---- full graph (symmetric: in-neighbours == CSR rows) ----
    in_off = indptr.to(torch.int32)
    deg = (indptr[1:] - indptr[:-1]).float() + 1.0
    dinv = deg.rsqrt()
    nnz = indices.numel()
    ref = None
    for v in (variants if os.environ.get("SKIP_FULL") is None else []):
        out, ms = run(L, g.ctx, x, F, None, N, in_off, indices, dinv, v)
        if ref is None:
            ref = out
        same = bool(torch.equal(out, ref))
        alg = 4.0 * N * F * 2 + 4.0 * nnz + 12.0 * N              # X read once + Y written once + indices + offsets/dinv
        gathered = 4.0 * F * (nnz + N) + 4.0 * N * F + 4.0 * nnz   # bytes the SMs actually pull (rows re-read per edge)
        res[f"full_v{v}"] = {"ms": round(ms, 3), "bitwise_equal_v0": same, "alg_GBps": round(alg / ms / 1e6, 1),
                             "gathered_GBps": round(gathered / ms / 1e6, 1)}
        print(f"full-graph v{v}: {ms:.3f} ms  equal={same}  algorithmic {alg/ms/1e6:.0f} GB/s  gathered {gathered/ms/1e6:.0f} GB/s", flush=True)
        del out
    del ref
    # ---- frontier-shaped: n sorted random rows, one source each among 1280 'prev' rows, output hi/lo at ldY ----
    n = 65000
    gen = torch.Generator(device=dev).manual_seed(1)
    nodes = torch.sort(torch.randperm(N, generator=gen, device=dev)[:n]).values.to(torch.int32)
    src = torch.randint(0, 1280, (n,), generator=gen, device=dev, dtype=torch.int32)
    src = torch.where(src == torch.arange(n, device=dev, dtype=torch.int32), src + 1, src)
    off = torch.arange(n + 1, device=dev, dtype=torch.int32)
    dv = torch.rand(n, generator=gen, device=dev) * 0.5 + 0.1
    ldo = ((F + 4 + 3) // 4) * 4
    ref = None
    for v in variants:
        out, ms = run(L, g.ctx, x, F, nodes, n, off, src, dv, v, reps=9, hi_lo=True, ldo=ldo)
        if ref is None:
            ref = out
        same = bool(torch.equal(out, ref))
        alg = 4.0 * n * (F + ldo) + 12.0 * n + 4.0 * n
        res[f"hop_v{v}"] = {"us": round(ms * 1e3, 2), "bitwise_equal_v0": same, "alg_GBps": round(alg / ms / 1e6, 1)}
        _, ms2 = run(L, g.ctx, x, F, nodes, n, off, src, dv, v, reps=9, hi_lo=False, ldo=ldo)
        _, ms3 = run(L, g.ctx, x, F, nodes, n, off, src, dv, v, reps=9, hi_lo=True, ldo=ldo, do_flush=False)
        print(f"hop-shaped v{v}: {ms*1e3:.2f} us  equal={same}  algorithmic {alg/ms/1e6:.0f} GB/s; single fp32 output {ms2*1e3:.2f} us; hi/lo warm L2 {ms3*1e3:.2f} us", flush=True)
    # ---- the engine's hop aggregation itself: indicator columns + ones column, (hi, lo) output ----
    bits = torch.randint(0, 16, (n,), generator=gen, device=dev, dtype=torch.int32)
    ldo2 = ((F + 4 + 1 + 3) // 4) * 4
    cnt = torch.tensor([n], dtype=torch.int32, device=dev)
    hi, lo = torch.zeros(n, ldo2, device=dev), torch.zeros(n, ldo2, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    flush = torch.zeros(256 << 20, dtype=torch.uint8, device=dev)
    keep = {}
    for v in variants:
        L.cdll.grapes_agg_variant(v)
        ts = []
        for it in range(12):
            flush.sum()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            L.grapes_aggregate(g.ctx, ptr(x), F, F, ptr(nodes), cnt.data_ptr(), n, ptr(off), ptr(src), ptr(dv), ptr(bits), 4,
                               None, 0, None, ldo2, ptr(hi), ptr(lo), F + 4, st)
            e1.record(); torch.cuda.synchronize()
            if it: ts.append(e0.elapsed_time(e1))
        ts.sort()
        keep[v] = (hi.clone(), lo.clone())
        alg = 4.0 * n * (F + ldo2) + 12.0 * n + 4.0 * n
        res[f"hop_ind_v{v}"] = {"us": round(ts[len(ts) // 2] * 1e3, 2), "alg_GBps": round(alg / ts[len(ts) // 2] / 1e6, 1)}
        print(f"hop aggregation with indicators v{v}: {ts[len(ts)//2]*1e3:.2f} us", flush=True)
    L.cdll.grapes_agg_variant(0)
    res["hop_ind_bitwise_equal"] = bool(torch.equal(keep[0][0], keep[1][0]) and torch.equal(keep[0][1], keep[1][1]))
    print(json.dumps(res))


if __name__ == "__main__":
    main()
