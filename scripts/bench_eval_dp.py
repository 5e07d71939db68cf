"""Data-parallel full-batch evaluation (grapes_b200.gcn.full_graph_forward_sharded) against the replicated one
(full_graph_forward_streamed on every rank), per rank.  Run under torchrun, one process per GPU (1 process is W = 1):

    torchrun --nproc-per-node 2 scripts/bench_eval_dp.py --shapes products papers --out profiles/r06_eval_dp_w2.json

Per shape and rank: window structure build ms, layer-1 ms, layer-2 ms (Z read from its owners over peer memory), the
bytes layer 2 gathers and the part of them that is remote, torch.cuda.max_memory_allocated; the same for the replicated
evaluation; and layer 2 after an NCCL all-gather of Z (the alternative that keeps all of Z on every rank).  Times are CUDA
events, the median of --reps runs after one warm-up run; the ranks are aligned by a barrier before each timed run.
Gathered bytes count every (self + source) row once: a floor of the traffic."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
GB = 1 << 30


def _timed(fn, reps, sync):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    ts = []
    for _ in range(reps):
        sync()
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
        return q
    except Exception as exc:                                   # reported, never fatal
        return f"unknown ({type(exc).__name__})"


def shape(name, reps, rank, world, dev):
    from bench import build_workload
    from grapes_b200.dist import PeerRowTable
    from grapes_b200.gcn import (GCN, LocalRowTable, ShardedGraphNorm, WideGraphNorm, full_graph_forward_streamed,
                                 sharded_layer1, sharded_layer2)
    from grapes_b200.graph import DeviceGraph
    sync = (lambda: dist.barrier()) if world > 1 else (lambda: None)
    cfg, indptr, indices, x, y, train_idx = build_workload(name, 0, dev)
    del train_idx
    N, F, C = cfg["N"], cfg["F"], cfg["C"]
    C4 = (C + 3) // 4 * 4
    graph = DeviceGraph(indptr, indices, N)
    torch.manual_seed(0)
    gcn_c = GCN(F, [256, C]).to(dev).eval()
    mask = torch.zeros(N, dtype=torch.bool, device=dev)
    mask[::97] = True
    res = {"nodes": N, "stored_edges": int(indices.numel()), "features": F, "feature_dtype": str(x.dtype), "classes": C,
           "resident_before_GB": torch.cuda.memory_allocated() / GB}

    # replicated: what every rank runs without a group
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    try:
        wn = WideGraphNorm(graph)
        ms = _timed(lambda: full_graph_forward_streamed(gcn_c, x, wn, y=y, mask=mask, return_logits=False), reps, sync)
        res["replicated"] = {"forward_ms": ms, "peak_allocated_GB": torch.cuda.max_memory_allocated() / GB}
        del wn
    except torch.OutOfMemoryError as exc:
        res["replicated"] = {"error": f"OutOfMemoryError: {exc}"[:300]}
    torch.cuda.empty_cache()

    # sharded
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    sgn = ShardedGraphNorm(graph, world, rank)
    e1.record()
    torch.cuda.synchronize()
    rows = max(sgn.bounds[r + 1] - sgn.bounds[r] for r in range(world))
    table = PeerRowTable(rows, C4, dev).rendezvous() if world > 1 else LocalRowTable.make(1, rows, C4, dev)[0]
    sh = {"bounds": sgn.bounds, "window_rows": sgn.rows, "window_nnz": sgn.E, "build_ms": e0.elapsed_time(e1),
          "build_peak_allocated_GB": torch.cuda.max_memory_allocated() / GB}
    remote = int(((sgn.in_src < sgn.lo) | (sgn.in_src >= sgn.hi)).sum()) if sgn.E else 0
    sh["layer2_gathered_GB"] = (sgn.E + sgn.rows) * C4 * 4 / 1e9
    sh["layer2_remote_GB"] = remote * C4 * 4 / 1e9
    sh["layer1_ms"] = _timed(lambda: sharded_layer1(gcn_c, x, sgn, table), reps, sync)
    sync()
    table.barrier()
    sh["layer2_ms"] = _timed(lambda: sharded_layer2(gcn_c, sgn, table, y=y, mask=mask), reps, sync)
    sh["layer2_gather_rate_GBps"] = sh["layer2_gathered_GB"] / (sh["layer2_ms"] / 1e3)
    sh["peak_allocated_GB"] = torch.cuda.max_memory_allocated() / GB
    if world > 1:
        # alternative: all-gather Z by NCCL, then the same kernel over local copies of every window
        gathered = torch.empty((world * table.rows.shape[0], C4), dtype=torch.float32, device=dev)
        local = type("T", (), {})()
        local.ld = C4
        local.ptrs = (ctypes.c_void_p * world)(*[gathered[o * table.rows.shape[0]:].data_ptr() for o in range(world)])

        def allgather_layer2():
            dist.all_gather_into_tensor(gathered, table.rows)
            sharded_layer2(gcn_c, sgn, local, y=y, mask=mask)
        sh["allgather_layer2_ms"] = _timed(allgather_layer2, reps, sync)
        sh["allgather_Z_GB_per_rank"] = gathered.numel() * 4 / GB
        sh["allgather_peak_allocated_GB"] = torch.cuda.max_memory_allocated() / GB
        del gathered
    res["sharded"] = sh
    del sgn, table, graph, indptr, indices, x
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", nargs="+", default=["products", "papers"])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    out = {"world": world, "gpu": _gpu(), "shapes": {}}
    try:
        for s in args.shapes:
            r = shape(s, args.reps, rank, world, dev)
            per_rank = [None] * world
            if world > 1:
                dist.all_gather_object(per_rank, r)
            else:
                per_rank = [r]
            out["shapes"][s] = per_rank
            if rank == 0:
                print(json.dumps({s: per_rank}), flush=True)
        if rank == 0 and args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                json.dump(out, f, indent=1)
    finally:
        if world > 1:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
