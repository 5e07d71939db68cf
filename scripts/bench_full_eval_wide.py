"""Full-batch evaluation on the int64 whole-graph structure and the row-slab forward (grapes_b200.gcn.WideGraphNorm,
full_graph_forward_streamed): the path evaluate(full_batch=True) takes from eval.WIDE_MIN_EDGES edges on.  Writes ONE JSON:

* papers shape (111 M nodes, 3.2 G stored edges, bf16 table; bench.build_workload("papers")): structure build time, the
  forward split into its layer-1 slabs and its layer-2 aggregation, torch.cuda.max_memory_allocated after each phase, the
  bytes each aggregation gathers and the rate that follows from them;
* products shape: the streamed path, forced, against the current GraphNorm path (gcn_c(x, GraphNorm)) on the same graph,
  and whether their logits are bit-identical.

    python scripts/bench_full_eval_wide.py --out profiles/r05_full_eval_wide.json

Times are CUDA events, the median of --reps runs after one warm-up run.  Gathered bytes count every (self + source) row an
aggregation reads once: (nnz + N) x row bytes; the tables are far larger than L2, so this is a floor of the DRAM traffic."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
HBM_DATASHEET_GBPS = 7700.0           # HGX B200 data sheet, one GPU


def _timed(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return sorted(ts)[len(ts) // 2]


def _gpu():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else None
    except Exception as exc:                                   # reported, never fatal
        return f"unknown ({type(exc).__name__})"


def _agg_all(gn, X, out, slabs, R, N):
    for i, r0 in enumerate(range(0, N, R)):
        gn.aggregate_rows(X, slabs[i], min(R, N - r0), out)


def papers(reps):
    from bench import build_workload
    from grapes_b200._lib import GrapesError
    from grapes_b200.gcn import GCN, WideGraphNorm, full_graph_forward_streamed
    from grapes_b200.graph import DeviceGraph
    dev = torch.device("cuda", 0)
    cfg, indptr, indices, x, y, train_idx = build_workload("papers", 0, dev)
    del train_idx
    N, F, C = cfg["N"], cfg["F"], cfg["C"]
    graph = DeviceGraph(indptr, indices, N)
    torch.manual_seed(0)
    gcn_c = GCN(F, [256, C]).to(dev).eval()
    GB = 1 << 30
    res = {"workload": "papers", "nodes": N, "stored_edges": int(indices.numel()), "features": F,
           "feature_dtype": str(x.dtype), "classes": C, "hidden": 256,
           "resident_before_GB": torch.cuda.memory_allocated() / GB}
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    gn = WideGraphNorm(graph)
    e1.record()
    torch.cuda.synchronize()
    res["structure"] = {"build_ms": e0.elapsed_time(e1), "nnz_without_self_loops": gn.E,
                        "in_off_last": int(gn.in_off[-1]), "peak_allocated_GB": torch.cuda.max_memory_allocated() / GB,
                        "resident_after_GB": torch.cuda.memory_allocated() / GB,
                        "note": "one-off, cached on the graph; includes the nnz read-back and the workspace allocation"}
    mask = torch.zeros(N, dtype=torch.bool, device=dev)
    mask[::97] = True
    free, total = torch.cuda.mem_get_info(dev)
    res["before_forward"] = {"device_free_GB": free / GB, "torch_allocated_GB": torch.cuda.memory_allocated() / GB,
                             "torch_reserved_GB": torch.cuda.memory_reserved() / GB,
                             "resident_Z_GB": N * ((C + 3) // 4 * 4) * 4 / GB,
                             "note": "device memory outside torch's allocator is the graph's library context (sized "
                                     "for frontiers of N nodes) and the CUDA context"}
    torch.cuda.reset_peak_memory_stats()
    try:
        fwd_ms = _timed(lambda: full_graph_forward_streamed(gcn_c, x, gn, y=y, mask=mask, return_logits=False), reps)
    except GrapesError as exc:
        res["forward"] = {"error": str(exc)}
        return res
    res["forward"] = {"ms": fwd_ms, "peak_allocated_GB": torch.cuda.max_memory_allocated() / GB,
                      "what": "full_graph_forward_streamed with masked scores, no [N, C] logits (evaluate's default)"}
    C4 = (C + 3) // 4 * 4
    try:
        _aggregations(res, gn, x, N, F, C, C4, fwd_ms, reps, dev)
    except (GrapesError, torch.OutOfMemoryError) as exc:
        res["aggregations"] = {"error": f"{type(exc).__name__}: {exc}"[:400]}
    res["peak_allocated_GB_all_phases"] = torch.cuda.max_memory_allocated() / GB
    res["device_total_GB"] = torch.cuda.get_device_properties(dev).total_memory / GB
    return res


def _aggregations(res, gn, x, N, F, C, C4, fwd_ms, reps, dev):
    """each aggregation of the forward alone, over the same slabs"""
    from grapes_b200.gcn import slab_rows_for
    R = slab_rows_for(N, 4 * (F + 256 + C4), N * C4 * 4, dev)
    slabs = torch.tensor([[min(R, N - r0), r0] for r0 in range(0, N, R)], dtype=torch.int32, device=dev)
    Y = torch.empty((R, F), dtype=torch.float32, device=dev)
    Z = torch.zeros((N, C4), dtype=torch.float32, device=dev)
    out = torch.empty((R, C4), dtype=torch.float32, device=dev)
    a1 = _timed(lambda: _agg_all(gn, x, Y, slabs, R, N), reps)
    a2 = _timed(lambda: _agg_all(gn, Z, out, slabs, R, N), reps)
    rows = gn.E + N
    b1, b2 = rows * F * x.element_size(), rows * C4 * 4
    res["slab_rows"] = R
    res["slabs"] = len(slabs)
    res["layer2_aggregation"] = {"ms": a2, "gathered_bytes": b2, "GBps": b2 / a2 / 1e6,
                                 "share_of_datasheet_hbm": b2 / a2 / 1e6 / HBM_DATASHEET_GBPS}
    res["layer1_slabs"] = {"ms": fwd_ms - a2, "aggregation_ms": a1, "gathered_bytes": b1, "aggregation_GBps": b1 / a1 / 1e6,
                           "aggregation_share_of_datasheet_hbm": b1 / a1 / 1e6 / HBM_DATASHEET_GBPS,
                           "gemm_flop": 2 * N * (F * 256 + 256 * C),
                           "note": "forward ms minus the layer-2 aggregation ms: slab aggregations, both SIMT GEMMs, relu"}


def products(reps):
    from bench import build_workload
    from grapes_b200.gcn import GCN, GraphNorm, WideGraphNorm, full_graph_forward_streamed
    from grapes_b200.graph import DeviceGraph
    dev = torch.device("cuda", 0)
    cfg, indptr, indices, x, y, train_idx = build_workload("products", 0, dev, native_csr=True)
    N, F, C = cfg["N"], cfg["F"], cfg["C"]
    graph = DeviceGraph(indptr, indices, N)
    torch.manual_seed(0)
    gcn_c = GCN(F, [256, C]).to(dev).eval()
    gn, wn = GraphNorm(graph), WideGraphNorm(graph)
    with torch.no_grad():
        cur_ms = _timed(lambda: gcn_c(x, gn), reps)
        ref = gcn_c(x, gn)[0]
    wide_ms = _timed(lambda: full_graph_forward_streamed(gcn_c, x, wn), reps)
    got, _ = full_graph_forward_streamed(gcn_c, x, wn)
    return {"workload": "products", "nodes": N, "stored_edges": int(indices.numel()), "features": F, "classes": C,
            "current_path_ms": cur_ms, "streamed_forced_ms": wide_ms, "logits_bit_identical": bool(torch.equal(got, ref)),
            "what": "gcn_c(x, GraphNorm) (int32 structure, whole-graph arrays) against full_graph_forward_streamed on "
                    "WideGraphNorm, both returning [N, C] logits"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--skip-papers", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_full_eval_wide.py measures on a CUDA device; none is available")
    out = {"gpu": _gpu(), "products": products(args.reps)}
    torch.cuda.empty_cache()
    if not args.skip_papers:
        out["papers"] = papers(args.reps)
    line = json.dumps(out, indent=1)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
