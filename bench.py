#!/usr/bin/env python
"""Benchmark of the GRAPES sample+train step (BASELINE.json metric: target nodes/sec).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port) on host cores

A "step" is one batch of the reference's training loop (main.py:161-291): 3-hop frontier expansion +
sampler GCN + Gumbel-top-k per hop, gcn_z, classifier forward/backward, GFlowNet loss backward, both
Adam updates.  Workload (N=1): the ogbn-products-shaped synthetic graph BASELINE.json's metric is quoted
on (2,449,029 nodes, 61.9M undirected pairs -> ~123.7M nnz, 100 features, 47 classes, batch 1024,
k=256/hop, 3 hops, hidden 256).  Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True      # the benchmark leaves the tree it runs from untouched (it may be read-only)
sys.path.insert(0, ROOT)
from grapes_b200.synth import SHAPES  # noqa: E402


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="grapes_b200", choices=["grapes_b200", "reference"])
    ap.add_argument("--workload", default="products", choices=list(SHAPES))
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of CUDA-graph replay")
    ap.add_argument("--no-spmm", action="store_true", help="skip the whole-graph SpMM leg")
    ap.add_argument("--exchange", default="peer", choices=["peer", "nccl", "none"],
                    help="N > 1: 'peer' = gradient scale + push all-reduce + Adam as ONE kernel over NVLink peer memory inside "
                         "the step graph (default); 'nccl' = ncclAllReduce(AVG) of the flat gradient captured into the step graph; "
                         "'none' = DIAGNOSTIC ONLY: the ranks train independent replicas (no exchange), to price the exchange")
    ap.add_argument("--prime", type=int, default=40, help="untimed steps before the W warm-up steps (clocks, allocator, graph variants, communicator)")
    ap.add_argument("--no-prefetch", action="store_true", help="no cross-step prefetch of the next batch's hop-0 front end")
    ap.add_argument("--cpu-budget-s", type=float, default=12.0)
    ap.add_argument("--full-eval", action="store_true",
                    help="also run scripts/bench_full_eval.py (full-graph evaluation forward on the opt-in tensor-core path, NOT yet "
                         "verified on a GPU) in a process of its own and attach its line as `full_graph_eval`")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed (losses, sampler statistics, sampled "
                         "nodes, classifier logits, updated parameters) as DIR/<name>.npy, to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "grapes_b200":
        ap.error("--dump-outputs writes the outputs of the grapes_b200 arm")
    return args


# --------------------------------------------------------------------------------------------
def build_workload(name: str, seed: int, device, native_csr: bool = False):
    """SURVEY.md section 8(d) generator on `device` (one-off, untimed).  native_csr=True (this repo's arm): the CSR is built
    by grapes_csr_from_edges (csrc/csr_build.cu, the replacement of main.py:134-136) and its event-timed duration is
    returned in cfg["csr_build"]; False (reference arm, may be a CPU-only process): torch sort/unique, same result."""
    cfg = dict(SHAPES[name])
    N, E_dir, F, C, n_train = cfg["N"], cfg["E_dir"], cfg["F"], cfg["C"], cfg["n_train"]
    g = torch.Generator(device=device).manual_seed(seed)
    if name == "papers":
        return build_workload_blocked(cfg, g, device)
    half = E_dir // 2
    src = torch.randint(0, N, (half,), generator=g, device=device, dtype=torch.int64)
    dst = torch.randint(0, N, (half,), generator=g, device=device, dtype=torch.int64)
    if native_csr:
        from grapes_b200.graph import csr_from_edge_index
        ei = torch.stack([torch.cat([src, dst]), torch.cat([dst, src])])
        del src, dst
        csr_from_edge_index(ei[:, :1024], N, device)            # load the library, warm the allocator
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        indptr, indices = csr_from_edge_index(ei, N, device)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        E, nnz = int(ei.shape[1]), int(indices.numel())
        alg = 16 * E + 4 * E + 16 * E + 8 * E + 8 * E + 4 * E + 8 * E + 2 * 12 * N + 8 * nnz   # phases listed in csrc/csr_build.cu
        cfg["csr_build"] = {"entry": "grapes_csr_from_edges", "edges_in": E, "nnz": nnz, "ms": ms,
                            "algorithmic_GBps": alg / ms / 1e6,
                            "note": "one-off (main.py:134-136; scipy on the host in the reference), includes workspace "
                                    "allocation and the nnz read-back"}
        del ei
    else:
        key = torch.cat([src * N + dst, dst * N + src])
        del src, dst
        key = torch.unique(key, sorted=True)                 # csr_matrix(bool) collapses duplicates (main.py:134)
        rows = torch.div(key, N, rounding_mode="floor")
        indices = (key - rows * N).to(torch.int32)
        del key
        counts = torch.bincount(rows, minlength=N)
        del rows
        indptr = torch.zeros(N + 1, dtype=torch.int64, device=device)
        torch.cumsum(counts, 0, out=indptr[1:])
    x = torch.randn(N, F, generator=g, device=device, dtype=torch.float32)
    y = torch.randint(0, C, (N,), generator=g, device=device, dtype=torch.int64)
    train_idx = torch.sort(torch.randperm(N, generator=g, device=device)[:n_train]).values
    return cfg, indptr, indices, x, y, train_idx


def build_workload_blocked(cfg, g, device, blocks: int = 64):
    """papers100M-shaped graph (111 M nodes, 3.2 G stored edges, 128 bf16 features; BASELINE.json configs[4]) built one
    row block at a time so the peak stays far below 180 GB: block b draws its share of directed edges with sources in
    its row range and uniform destinations, sorts + collapses duplicates (the CSR constructor of main.py:134-136) and
    appends to the preallocated int32 `indices`.  Directed, not symmetrised (a global symmetrisation needs a 3.2 G-key
    sort); indptr is int64 and exceeds 2^31.  Features are drawn per block and stored as bf16."""
    N, E_dir, F, C, n_train = cfg["N"], cfg["E_dir"], cfg["F"], cfg["C"], cfg["n_train"]
    indices = torch.empty(E_dir, dtype=torch.int32, device=device)
    counts = torch.zeros(N, dtype=torch.int64, device=device)
    x = torch.empty(N, F, dtype=torch.bfloat16, device=device)
    rows_per = (N + blocks - 1) // blocks
    filled = 0
    for b in range(blocks):
        r0, r1 = b * rows_per, min(N, (b + 1) * rows_per)
        if r0 >= r1:
            break
        m = int(round(E_dir * (r1 - r0) / N))
        src = torch.randint(r0, r1, (m,), generator=g, device=device, dtype=torch.int64)
        dst = torch.randint(0, N, (m,), generator=g, device=device, dtype=torch.int64)
        key = torch.unique(src * N + dst, sorted=True)
        del src, dst
        rows = torch.div(key, N, rounding_mode="floor")
        indices[filled:filled + key.numel()] = (key - rows * N).to(torch.int32)
        counts[r0:r1] = torch.bincount(rows - r0, minlength=r1 - r0)
        filled += int(key.numel())
        del key, rows
        x[r0:r1] = torch.randn(r1 - r0, F, generator=g, device=device, dtype=torch.float32).to(torch.bfloat16)
    indices = indices[:filled].clone() if filled < E_dir * 0.98 else indices[:filled]
    indptr = torch.zeros(N + 1, dtype=torch.int64, device=device)
    torch.cumsum(counts, 0, out=indptr[1:])
    del counts
    y = torch.randint(0, C, (N,), generator=g, device=device, dtype=torch.int64)
    train_idx = torch.sort(torch.randperm(N, generator=g, device=device)[:n_train]).values
    cfg["E_stored"] = filled
    return cfg, indptr, indices, x, y, train_idx


class ClockSampler:
    """Samples SM clocks / throttle reasons DURING the timed region: NVML polled every 1 ms from a thread
    (B200_PROFILING.md clocks line; nvidia-smi -lms is too coarse for a 20 ms region and is only the fallback)."""
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index: int):
        self.index, self.trace, self.stop_flag, self.thread = index, [], False, None
        self.t0 = self.t1 = None
        self.max_mhz, self.nvml, self.handle = None, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = index
            if visible:
                ids = [v.strip() for v in visible.split(",") if v.strip()]
                if index < len(ids) and ids[index].isdigit():
                    phys = int(ids[index])
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _poll(self):
        nv = self.nvml
        bits = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        while not self.stop_flag:
            try:
                t = time.perf_counter()
                mhz = float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                self.trace.append((t, mhz, [name for name, bit in bits.items() if r & bit]))
            except Exception:
                pass
            time.sleep(0.0005)

    def start(self):
        """The polling thread starts BEFORE the warm-up (its first NVML calls take milliseconds); only the samples between
        mark_begin() and mark_end() -- the timed region -- are reported."""
        if self.nvml is None:
            return
        self.trace, self.t0, self.t1 = [], None, None
        self.thread = threading.Thread(target=self._poll, daemon=True)
        self.thread.start()

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        if self.nvml is None:
            return self._smi_once()
        self.stop_flag = True
        self.thread.join(timeout=1.0)
        t0 = self.t0 if self.t0 is not None else 0.0
        t1 = self.t1 if self.t1 is not None else float("inf")
        inside = [e for e in self.trace if t0 <= e[0] <= t1]
        if not inside and self.trace:                     # a window shorter than one poll: the samples around it
            inside = sorted(self.trace, key=lambda e: min(abs(e[0] - t0), abs(e[0] - t1)))[:2]
        sm = sorted(e[1] for e in inside)
        reasons = sorted({n for e in inside for n in e[2]})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "samples": len(sm),
                "reasons": reasons, "source": "nvml, polled every ~0.5 ms from before the warm-up; samples inside the timed region"}

    def _smi_once(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                 capture_output=True, text=True, timeout=10).stdout.strip().split(",")
            reasons = [n for n, v in zip(self.NAMES, out[2:6]) if v.strip().lower().startswith("active")]
            return {"sm_mhz": float(out[0]), "sm_max_mhz": float(out[1]), "samples": 1, "reasons": reasons,
                    "source": "nvidia-smi after the timed region (NVML unavailable)"}
        except Exception:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["nvidia-smi unavailable"]}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops_sustained", 1400.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, 1400.0, "fallback (B200_PROFILING.md)"


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(eng, out_dir: str):
    """Writes what the engine's last step handed back to its caller as ``out_dir/<name>.npy``: the losses and the per-hop
    sampler statistics main.py logs, the nodes sampled at each hop, the batch's nodes with the classifier's logits over
    them, the three networks' parameters after the optimiser update and the two optimisers' step counts (every step the
    engine ran, untimed ones included).  Floats stay float32; node ids are stored as
    float64 (exact).  The workload and every random draw are functions of the command-line seed, so two builds run with
    the same arguments can be compared file by file."""
    import numpy as np
    from grapes_b200.engine import SCAL
    torch.cuda.synchronize()
    scal = eng.scal.cpu().double()
    out = {k: scal[SCAL[k]:SCAL[k] + 1] for k in ("loss_c", "loss_gfn", "log_z", "tot_log_prob")}
    out["sampler_stats"] = eng.stats.cpu()
    for h, sz in enumerate(eng.hop_sizes()):
        out[f"sampled_hop{h}"] = eng.prev[h + 1][eng.bsz:eng.bsz + sz["s"]].cpu().double()
    A = eng.count("A")
    out["all_nodes"] = eng.all_nodes[:A].cpu().double()
    out["logits_c"] = eng.logits_c[:A].cpu()
    out["adam_steps"] = eng.adam_steps.cpu()
    for net, params in eng.state_dicts().items():
        for name, t in params.items():
            out[f"{net}.{name}"] = t.cpu()
    arrays = {k: v.numpy() for k, v in out.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (k, a.dtype)
        np.save(os.path.join(out_dir, k + ".npy"), a)


# --------------------------------------------------------------------------------------------
def cpu_reference_run(cfg, indptr, indices, x, y, train_idx, steps, warmup, budget_s, rank_offset=0):
    """Times the reference's CPU path (oracle port of main.py:161-291 + restated PyG GCNConv, torch CPU
    fp32, Adam) on the host cores.  Bounded: stops early once `budget_s` of timed work is spent."""
    import numpy as np
    import scipy.sparse as sp
    from oracle import reference_port as rp
    from grapes_b200.synth import SynthData
    torch.set_num_threads(os.cpu_count() or 1)
    N = cfg["N"]
    ip, ix = indptr.cpu().numpy(), indices.cpu().numpy()
    adj = sp.csr_matrix((np.ones(ix.shape[0], dtype=bool), ix, ip), shape=(N, N))
    data = SynthData(x=x.cpu(), y=y.cpu(), edge_index=torch.zeros(2, 0, dtype=torch.long), train_mask=None,
                     val_mask=None, test_mask=None, num_nodes=N, num_features=cfg["F"], num_classes=cfg["C"])
    st = rp.OracleState(data, sampling_hops=cfg["sampling_hops"], num_samples=cfg["num_samples"], hidden_dim=256,
                        seed=0, adjacency=adj)
    tr = train_idx.cpu()
    B = cfg["batch_size"]
    nb = tr.numel() // B
    done, t_total = 0, 0.0
    for j in range(warmup + steps):
        b = (rank_offset + j) % nb
        t0 = time.perf_counter()
        rp.reference_step(st, tr[b * B:(b + 1) * B])
        dt = time.perf_counter() - t0
        if j >= warmup:
            done += 1
            t_total += dt
            if t_total > budget_s:
                break
    return done, t_total, torch.get_num_threads()


_REAL_STDOUT = None


def emit(line: dict):
    """The ONE JSON line goes to the real stdout; everything else any library writes to fd 1 (NCCL prints its
    version banner there) was re-routed to stderr by main()."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    args = parse_args()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cfgname = args.workload
    have_cuda = torch.cuda.is_available()

    # ------------------------------------------------------------------ reference arm
    if args.impl == "reference":
        if rank != 0:
            return 0
        dev = torch.device("cuda", local_rank) if have_cuda else torch.device("cpu")
        cfg, indptr, indices, x, y, train_idx = build_workload(cfgname, args.seed, dev)
        warm = args.warmup
        done, t_total, threads = cpu_reference_run(cfg, indptr, indices, x, y, train_idx, args.steps, warm,
                                                   budget_s=150.0)
        B = cfg["batch_size"]
        val = done * B / t_total
        sample = f"{done} of the requested {args.steps} steps of batch {B} (stops after 150 s of timed work), {warm} warm-up"
        line = {"impl": "reference", "metric": "target nodes/sec (sample+train)", "value": val, "unit": "nodes/s",
                "n_gpus": args.gpus, "steps": done, "warmup": warm, "ms_per_step": 1e3 * t_total / done,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": workload_config(cfgname, cfg, 1),
                "cpu_baseline": {"value": val, "unit": "nodes/s", "cores": threads, "kind": "port", "sample": sample},
                "e2e": {"value": val, "unit": "nodes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        emit(line)
        return 0

    # ------------------------------------------------------------------ this repo's CUDA path
    if not have_cuda:
        print("bench.py: no CUDA device -- grapes_b200 has no CPU fallback", file=sys.stderr)
        return 2
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    from grapes_b200._lib import lib
    from grapes_b200.engine import GrapesEngine
    from grapes_b200.graph import DeviceGraph

    cfg, indptr, indices, x, y, train_idx = build_workload(cfgname, args.seed, dev, native_csr=True)
    csr_build = cfg.pop("csr_build", None)
    N, F, C, B = cfg["N"], cfg["F"], cfg["C"], cfg["batch_size"]
    graph = DeviceGraph(indptr, indices, N)
    eng = GrapesEngine(graph, x, y, num_classes=C, batch_size=B, num_samples=cfg["num_samples"],
                       sampling_hops=cfg["sampling_hops"], hidden_dim=256, seed=args.seed)
    L = lib()
    K, W = args.steps, max(args.warmup, 3)
    PRIME = max(args.prime, 0)
    nb = train_idx.numel() // B
    from grapes_b200.dist import shard_batches
    mine = shard_batches(nb, rank, world)                             # batch i -> rank i mod W
    order = [mine[j % len(mine)] for j in range(W + K + 1)]
    batches = torch.stack([train_idx[b * B:(b + 1) * B] for b in order]).to(torch.int32)
    use_graph = not args.no_graph
    prefetch = not args.no_prefetch
    # N > 1: the engine owns the exchange (GrapesEngine.enable_data_parallel): ONE collective per step, the mean of the
    # flat gradient (91 k floats on products-shape), fused with the gradient scale and both Adam updates into the step's
    # last launch over NVLink peer memory ('peer'), or ncclAllReduce captured into the step graph ('nccl').  Either way a
    # step is one graph launch and every rank ends it with bit-identical parameters.
    exchange_used = "none"
    if world > 1 and args.exchange != "none":
        eng.enable_data_parallel(exchange=args.exchange)
        exchange_used = "peer" if eng.peer is not None else "nccl"     # (peer falls back to nccl, on every rank, without P2P)

    def one_step(j):
        # the ids of batch j+1 are handed over with batch j: its reset + weight-independent hop-0 front end are enqueued
        # next to this step's classifier tail (the reference's DataLoader order is known in advance, main.py:125-126)
        nxt = batches[j + 1] if prefetch else None
        eng.step(batches[j], apply_optim=True, use_graph=use_graph, next_targets=nxt)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for j in range(PRIME):                                            # untimed: clocks up, every graph variant captured,
        one_step(j % W)                                               # communicator channels set up
    sync_all()
    sampler = ClockSampler(local_rank)
    sampler.start()
    for j in range(W):
        one_step(j)
    sync_all()
    eng.check_overflow()
    launches0 = L.grapes_kernel_launches()
    sync_all()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
    sampler.mark_begin()
    ev[0].record()
    for j in range(W, W + K):
        one_step(j)
        ev[j - W + 1].record()
    torch.cuda.synchronize()
    sampler.mark_end()
    sync_all()
    clocks = sampler.stop()
    ms = ev[0].elapsed_time(ev[K])
    eng.check_overflow()
    if args.dump_outputs and rank == 0:
        dump_outputs(eng, args.dump_outputs)         # before the e2e and profiling steps below overwrite them
    if use_graph:
        # kernels recorded into the graph once, replayed K times (the NCCL exchange adds its own all-reduce kernel)
        per_step = eng.launches_per_graph + (1 if exchange_used == "nccl" else 0)
        launches = per_step * K
    else:
        launches = L.grapes_kernel_launches() - launches0
        per_step = launches // K
    # per-step device times of this rank (event to event), gathered from every rank
    per = sorted(ev[i].elapsed_time(ev[i + 1]) for i in range(K))
    mine_t = torch.tensor([ms, per[len(per) // 2], per[min(len(per) - 1, int(0.99 * len(per)))], per[-1], per[0]], device=dev)
    if world > 1:
        allt = [torch.zeros_like(mine_t) for _ in range(world)]
        dist.all_gather(allt, mine_t)
    else:
        allt = [mine_t]
    step_times = [{"rank": r, "total_ms": float(t_[0]), "p50_ms": float(t_[1]), "p99_ms": float(t_[2]),
                   "max_ms": float(t_[3]), "min_ms": float(t_[4])} for r, t_ in enumerate(allt)]
    ms = max(st_["total_ms"] for st_ in step_times)                   # max over ranks
    value = world * B * K / (ms / 1e3)

    # ------------------------------------------------------------------ e2e: host buffers in, loss out, every step
    host_targets = torch.stack([train_idx[b * B:(b + 1) * B] for b in order]).to(torch.int64).cpu().pin_memory()
    host_scal = [torch.zeros(16, dtype=torch.float32).pin_memory() for _ in range(2)]
    scal_ready = [torch.cuda.Event(), torch.cuda.Event()]
    # ids: the loader's int64 batch (pinned host memory) is narrowed to int32 on the host and copied with ONE cudaMemcpyAsync
    # straight into the engine's target list of the step state that will run it (engine.set_targets accepts a pinned host
    # tensor) -- no staging buffer, no conversion kernel on the stream.  Three host slots: a slot is rewritten three steps
    # later, after the host has waited on the event of the step that consumed it.
    host_ids32 = [torch.zeros(B, dtype=torch.int32).pin_memory() for _ in range(3)]

    def h2d_ids(j):
        host_ids32[j % 3].copy_(host_targets[j])                                         # host: int64 -> int32
        return host_ids32[j % 3]                                                         # H2D happens in engine.set_targets

    e2e_state = {"have": -1, "pending": None, "losses": 0}

    def e2e_collect():
        """host read of the PREVIOUS step's losses: waits on that step's own event, so the device already runs the
        step enqueued after it (the two step states keep their scalar blocks apart)"""
        j = e2e_state["pending"]
        if j is not None:
            scal_ready[j % 2].synchronize()
            e2e_state["losses"] += 1
            e2e_state["last_loss"] = float(host_scal[j % 2][0])
            eng.raise_on_flags(int(host_scal[j % 2][15]))                                # frontier overflow / peer failure of THAT step
            e2e_state["pending"] = None

    def e2e_step(j):
        # every step copies ONE batch of ids host -> device (the next batch's when prefetching: its front end runs next to
        # this step's classifier tail) and reads the losses back on the host (main.py:269,291 loss.item()), one step
        # behind: step j is enqueued, then the host waits for step j-1's losses while the device works on step j
        cur = host_ids32[j % 3] if e2e_state["have"] == j else h2d_ids(j)
        nxt = None
        if prefetch:
            nxt = h2d_ids(j + 1)
            e2e_state["have"] = j + 1
        eng.step(cur, apply_optim=True, use_graph=use_graph, next_targets=nxt)
        host_scal[j % 2].copy_(eng.scal, non_blocking=True)                              # D2H: losses (+ overflow bits) of step j
        scal_ready[j % 2].record()
        e2e_collect()                                                                    # losses of step j - 1
        e2e_state["pending"] = j

    for j in range(3):
        e2e_step(j)
    e2e_collect()
    sync_all()
    e2e_state["losses"] = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for j in range(W, W + K):
        e2e_step(j)
    e2e_collect()                                                                        # the last step's losses: inside the timed region
    e1.record()
    sync_all()
    assert e2e_state["losses"] == K and e2e_state["last_loss"] == e2e_state["last_loss"]   # every step's loss reached the host
    t = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = float(t.item())
    e2e = {"value": world * B * K / (e2e_ms / 1e3), "unit": "nodes/s", "h2d_bytes_per_step": B * 4,
           "d2h_bytes_per_step": 64, "ms_per_step": e2e_ms / K,
           "readback": "every step's 64-byte loss block is copied to pinned host memory and read by the host one step "
                       "behind (per-step event), so the device is never idle while the host reads"}

    # ------------------------------------------------------------------ per-kernel breakdown + roofline (rank 0)
    line = None
    if rank == 0:
        hbm_peak, tf_peak, peak_src = load_peaks()
        P_STEPS = 5
        eng.multi_stream = False             # one stream: each kernel is timed alone, not against its co-runners
        eng.peer = eng.dp_group = None       # rank 0 alone from here on: local Adam, no exchange
        if eng.ctx_a is not graph.ctx:
            L.grapes_ctx_set_sm_limit(eng.ctx_a, 0)    # ... and with the whole GPU (in the step the backward branch is given 96 SMs)
        L.profiling = True                   # (after the host-only call above: it is not a kernel)
        per_hop_acc = None
        for j in range(P_STEPS):
            eng.set_targets(batches[j])
            # park the GPU for ~2 ms so the whole step is queued before it starts: the per-call CUDA events then
            # bracket device time only (no CPU launch gaps inside the brackets)
            torch.cuda._sleep(4_000_000)
            eng.step(None, apply_optim=True, use_graph=False)
            torch.cuda.synchronize()
            hs = eng.hop_sizes()
            if per_hop_acc is None:
                per_hop_acc = [{k: 0.0 for k in ("m", "n", "c", "nnz")} for _ in hs]
            for acc, h in zip(per_hop_acc, hs):
                for k in acc:
                    acc[k] += h[k] / P_STEPS
        prof = L.profile_summary()
        L.profiling = False
        eng.multi_stream = True
        per_hop = per_hop_acc
        H = cfg["sampling_hops"]
        breakdown = {k: round(v[0] / P_STEPS, 4) for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])}
        Fp, ldY, D = eng.Fp, eng.ldY, eng.D
        n_sum = sum(h["n"] for h in per_hop)
        nnz_sum = sum(h["nnz"] for h in per_hop)
        # algorithmic bytes / flops per STEP of each hot entry point (DESIGN.md section 5)
        fwd_flops = 2.0 * (n_sum * Fp * D + per_hop[0]["n"] * F * D)
        alg = {
            "grapes_aggregate": ("hbm", sum(4 * h["n"] * (F + ldY) + 12 * h["n"] + 4 * h["nnz"] for h in per_hop)),
            "grapes_sampler_l1_fwd": ("tensor", fwd_flops),
            "grapes_sampler_l1_bwd": ("tensor", 2.0 * fwd_flops),
            # tcgen05 path: the backward is ONE contraction S = mask^T (dz * Y) (no recompute), same flops as the forward
            "grapes_sampler_l1_fwd_tc": ("tensor", fwd_flops),
            "grapes_sampler_l1_bwd_tc": ("tensor", fwd_flops),
        }
        # DRAM traffic per launch (dram__bytes_read.sum + dram__bytes_write.sum) of the hop-level launches, from the
        # committed summary of the latest `ncu --set full` capture of this same command (profiles/ncu_traffic.json names
        # the commit and the report it was read from); null when the workload has no capture
        ncu_traffic, traffic_src = {}, None
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.isfile(tpath):
            tj = json.load(open(tpath))
            if tj.get("workload") == cfgname:
                ncu_traffic = tj.get("bytes_per_launch", {})
                traffic_src = {k: tj.get(k) for k in ("commit", "report", "command")}
        rooflines = {}
        for name, (bound, work) in alg.items():
            if name not in prof:
                continue
            sec = prof[name][0] / P_STEPS / 1e3
            calls = prof[name][1] / P_STEPS
            if bound == "hbm":
                ach = work / sec / 1e9
                rooflines[name] = {"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                                   "frac": ach / hbm_peak, "traffic": ncu_traffic.get(name), "ms_per_step": sec * 1e3,
                                   "launches_per_step": calls, "algorithmic_bytes_per_launch": work / calls}
            else:
                ach = work / sec / 1e12
                rooflines[name] = {"bound": "tensor", "achieved": ach, "peak": tf_peak, "unit": "TFLOP/s",
                                   "frac": ach / tf_peak, "traffic": ncu_traffic.get(name), "ms_per_step": sec * 1e3,
                                   "launches_per_step": calls, "algorithmic_flops_per_launch": work / calls,
                                   "ceiling_frac": 1.0 / 6.0,
                                   "note": "3xTF32 (fp32-accurate): 3 tf32 MMAs per product at half the bf16 rate of the peak"}
        dominant = max(rooflines, key=lambda k: rooflines[k]["ms_per_step"]) if rooflines else None
        roof = dict(rooflines[dominant], kernel=dominant, peak_source=peak_src, traffic_source=traffic_src) if dominant else None

        # ---- whole-graph SpMM (the metric's "SpMM HBM GB/s"): Y = A_hat X over every edge of the workload graph, the
        # aggregation of the full-batch evaluation forward (eval.py:47-56); one launch of the TMA-staged kernel ----
        spmm, full_eval = None, None
        if world == 1 and not args.no_spmm and graph.nnz < (1 << 31) - 1:
            from grapes_b200.gcn import GraphNorm
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            gn = GraphNorm(graph)                    # one-off: gcn_norm structure of the whole graph
            ysp = gn.aggregate(x)
            torch.cuda.synchronize()
            ts = []
            for _ in range(5):
                s0.record()
                ysp = gn.aggregate(x)
                s1.record()
                torch.cuda.synchronize()
                ts.append(s0.elapsed_time(s1))
            ts.sort()
            sp_ms = ts[len(ts) // 2]
            nnz_g = int(gn.in_src.numel())
            alg_b = 4.0 * N * F * 2 + 4.0 * nnz_g + 12.0 * N          # X read once, Y written once, indices, offsets + deg^-1/2
            gat_b = 4.0 * F * (nnz_g + N) + 4.0 * N * F + 4.0 * nnz_g  # bytes the SMs pull: one feature row per edge and self-loop
            spmm = {"kernel": "k_agg_tma (grapes_aggregate)", "rows": N, "nnz": nnz_g, "width": F, "ms": sp_ms,
                    "algorithmic_GBps": alg_b / sp_ms / 1e6, "gathered_GBps": gat_b / sp_ms / 1e6,
                    "peak_GBps": hbm_peak, "frac_algorithmic": alg_b / sp_ms / 1e6 / hbm_peak,
                    "frac_gathered": gat_b / sp_ms / 1e6 / hbm_peak,
                    "note": "uniform-random graph: every edge gathers a 4F-byte row from a table 8x larger than L2, so the "
                            "traffic is the gathered bytes, not the algorithmic ones"}
            del ysp, gn

        cpu = None
        if world == 1 and not args.no_cpu_baseline and cfgname != "papers":      # the papers-shaped graph does not fit the host oracle
            done, t_total, threads = cpu_reference_run(cfg, indptr, indices, x, y, train_idx, 10, 1, args.cpu_budget_s)
            cpu = {"value": done * B / t_total, "unit": "nodes/s", "cores": threads, "kind": "port",
                   "sample": f"{done} steps of batch {B} on the same graph (oracle port of main.py:161-291, torch CPU fp32)",
                   "ms_per_step": 1e3 * t_total / done}
        # ---- full-graph evaluation forward gcn_c(x, edge_index) (eval.py:47-56; next-row f1) beside the oracle's CPU forward.
        # Written after this round's GPU budget was spent and never run on a GPU: only on request (--full-eval), and in its OWN
        # process (own CUDA context) so that whatever happens there costs this entry, never the bench line ----
        if world == 1 and args.full_eval and cfgname != "papers":
            try:
                cmd = [sys.executable, os.path.join(ROOT, "scripts", "bench_full_eval.py"), "--workload", cfgname,
                       "--seed", str(args.seed)] + (["--no-cpu"] if args.no_cpu_baseline else [])
                res = subprocess.run(cmd, capture_output=True, text=True, timeout=240)
                lines = [l for l in res.stdout.splitlines() if l.startswith("{")]
                full_eval = json.loads(lines[-1]) if (res.returncode == 0 and lines) else \
                    {"error": f"rc={res.returncode}: " + (res.stderr or res.stdout)[-300:]}
            except Exception as exc:                  # noqa: BLE001 -- reported, never hidden
                full_eval = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        line = {"metric": "target nodes/sec (sample+train)", "value": value, "unit": "nodes/s", "n_gpus": world,
                "steps": K, "warmup": W, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(cfgname, cfg, world),
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "launches_per_step": int(per_step),
                "roofline": roof, "rooflines": rooflines, "spmm": spmm, "full_graph_eval": full_eval, "csr_build": csr_build, "cpu_baseline": cpu, "breakdown_ms_per_step": breakdown,
                "frontier": per_hop, "cuda_graph": use_graph, "cross_step_prefetch": prefetch,
                "step_times": step_times, "prime_steps": PRIME,
                "gradient_exchange": ("none" if world == 1 else "NONE (diagnostic run: independent replicas, not data parallel)" if args.exchange == "none" else
                                      ("gradient scale + push all-reduce over NVLink peer memory + Adam: one kernel inside the step graph"
                                       if exchange_used == "peer" else "ncclAllReduce(AVG) captured into the step graph + Adam launch"))}
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def workload_config(name, cfg, world):
    sym = "directed, drawn per row block, duplicates collapsed" if name == "papers" else "symmetrised, duplicates collapsed"
    fbytes = 2 if name == "papers" else 4
    gb = (4.0 * cfg["E_dir"] + 8.0 * cfg["N"] + fbytes * cfg["N"] * cfg["F"]) / 1e9
    return {"workload": f"{name}-shaped synthetic graph: N={cfg['N']}, directed pairs={cfg['E_dir']} ({sym}), "
                        f"F={cfg['F']}, C={cfg['C']}, batch={cfg['batch_size']}, "
                        f"k={cfg['num_samples']}/hop, hops={cfg['sampling_hops']}, hidden=256, TB loss, Adam",
            "feature_storage": "bf16 (compute fp32)" if name == "papers" else "fp32",
            "global_batch": cfg["batch_size"] * world, "parallelism": f"dp{world} (targets sharded, graph+features replicated)",
            "l2_policy": f"inputs larger than L2: {gb:.1f} GB graph+features resident in HBM, every step gathers a different "
                         "frontier (tens of thousands of random rows per hop); no explicit flush"}


if __name__ == "__main__":
    sys.exit(main())
