"""A learned node-feature table sharded by rows with its Adam moments (dist.ShardedEmbedding) against the replicated
learned table, node_emb_dim = 64.

    python scripts/bench_embed_sharded.py --out result.json [--shapes products,papers] [--worlds 2,8]

One GPU, one process:
  * the table walk of one rank, grapes_adam_embed_rows over rows [0, ceil(N / W)) for W = 1, 2, 4, 8, against the
    whole-table grapes_adam_embed, products and papers row counts.  Every moment is non-zero (the dense walk reads and
    writes table, exp_avg and exp_avg_sq of every row: 24 N F / W bytes, plus 4096 gradient rows left out of the
    count); the tables are far larger than L2.  The forms
    alternate within each round, CUDA events around `--reps` launches, median over `--rounds` rounds;
  * ms/step of graph-replayed steps of the products-shaped engine with W = 4 emulated shards (it runs all W walks, so
    this is the overhead of the sharded path, not its gain) against the replicated learned-table engine, alternating.
Under torch.distributed.run, for each world size in --worlds the box has GPUs for: ms/step p50 / p99 per rank and table +
moment bytes per rank, replicated and sharded (peer exchange).  Other world sizes are reported as not measured.
The GPU name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ROWS = {"products": 2_449_029, "papers": 111_059_956}


def pct(v, q):
    v = sorted(v)
    return v[min(len(v) - 1, int(round(q / 100.0 * (len(v) - 1))))]


def gpu_info():
    import torch
    out = {"gpu": torch.cuda.get_device_name(0), "gpus_on_box": torch.cuda.device_count()}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        out["power_limit_and_max_sm_clock"] = q[0] if q else "unknown"
    except Exception as exc:                           # noqa: BLE001
        out["power_limit_and_max_sm_clock"] = f"unknown ({exc})"
    return out


def walk_bench(a):
    import torch
    from grapes_b200._lib import lib
    from grapes_b200.graph import DeviceGraph
    L, dev, F = lib(), torch.device("cuda", 0), 64
    out = {}
    for shape in a.shapes.split(","):
        N = ROWS[shape]
        g = DeviceGraph.from_edge_index(torch.tensor([[0], [1]]), N, device=dev, max_frontier=64)
        gen = torch.Generator(device=dev).manual_seed(0)
        x = torch.randn(N, F, generator=gen, device=dev)
        m = torch.randn(N, F, generator=gen, device=dev) * 1e-3
        v = torch.rand(N, F, generator=gen, device=dev) * 1e-6
        ids = torch.sort(torch.randperm(N, device=dev)[:4096]).values.to(torch.int32)
        words = (N + 31) // 32
        bm = torch.zeros(words, dtype=torch.int32, device=dev)
        bm.view(-1).index_put_((ids.long() >> 5,), (1 << (ids.long() & 31)).to(torch.int32), accumulate=True)
        pref = torch.zeros(words + 1, dtype=torch.int32, device=dev)
        pref[1:] = torch.cumsum(torch.bitwise_and(bm.view(-1, 1).bitwise_right_shift(torch.arange(32, device=dev)),
                                                  1).sum(1), 0).to(torch.int32)
        grows = torch.randn(4096, F, generator=gen, device=dev) * 1e-2
        steps = torch.full((2,), 10.0, device=dev)
        st = torch.cuda.current_stream().cuda_stream
        common = (F, bm.data_ptr(), pref.data_ptr(), grows.data_ptr(), F, 1e-3, 0.9, 0.999, 1e-8, steps.data_ptr(), st)
        forms = {"whole": lambda: L.grapes_adam_embed(g.ctx, x.data_ptr(), m.data_ptr(), v.data_ptr(), N, *common)}
        for W in (1, 2, 4, 8):
            rows = -(-N // W)
            forms[f"rows_W{W}"] = (lambda rows=rows: L.grapes_adam_embed_rows(
                g.ctx, x.data_ptr(), m.data_ptr(), v.data_ptr(), N, 0, rows, *common))
        for f in forms.values():
            f()
        torch.cuda.synchronize()
        times = {k: [] for k in forms}
        for _ in range(a.rounds):
            for k, f in forms.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(a.reps):
                    f()
                e1.record()
                torch.cuda.synchronize()
                times[k].append(e0.elapsed_time(e1) / a.reps)
        res = {}
        for k, t in times.items():
            rows = N if k == "whole" else -(-N // int(k.split("W")[1]))
            ms = pct(t, 50)
            res[k] = {"rows": rows, "ms_p50": ms, "ms_min": min(t), "bytes": 24 * rows * F,
                      "GB_per_s": 24 * rows * F / (ms * 1e6)}
        out[shape] = res
        print(shape, json.dumps(res), flush=True)
        del x, m, v, g
        torch.cuda.empty_cache()
    return out


def engine_bench(a):
    import torch
    from bench import build_workload
    from grapes_b200.dist import ShardedEmbedding
    from grapes_b200.engine import GrapesEngine
    from grapes_b200.graph import DeviceGraph
    dev = torch.device("cuda", 0)
    cfg, indptr, indices, _x, y, train_idx = build_workload("products", 0, dev, native_csr=True)
    del _x
    N, B = cfg["N"], cfg["batch_size"]
    g = DeviceGraph(indptr, indices, N)
    table = torch.randn(N, 64, generator=torch.Generator(device=dev).manual_seed(0), device=dev)
    hp = dict(num_classes=cfg["C"], batch_size=B, num_samples=cfg["num_samples"], sampling_hops=cfg["sampling_hops"],
              embed_nodes=True, seed=0)
    W = 4
    engines = {"replicated": GrapesEngine(g, table.clone(), y, **hp),
               f"emulated_W{W}": GrapesEngine(g, ShardedEmbedding.emulate(table, W)[0], y, **hp)}
    batches = [b.to(torch.int32).contiguous() for b in torch.split(train_idx, B) if b.numel() == B]
    for eng in engines.values():
        for i in range(a.warmup):
            eng.step(batches[i % len(batches)], use_graph=True)
    torch.cuda.synchronize()
    times = {k: [] for k in engines}
    for r in range(a.rounds):
        for k, eng in engines.items():
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(a.steps + 1)]
            ev[0].record()
            for i in range(a.steps):
                eng.step(batches[(r * a.steps + i) % len(batches)], use_graph=True)
                ev[i + 1].record()
            torch.cuda.synchronize()
            eng.check_overflow()
            times[k] += [ev[i].elapsed_time(ev[i + 1]) for i in range(a.steps)]
    res = {k: {"ms_per_step_p50": pct(t, 50), "ms_per_step_p99": pct(t, 99), "steps": len(t)} for k, t in times.items()}
    print("engine", json.dumps(res), flush=True)
    return res


def dp_worker(a):
    import torch
    import torch.distributed as dist
    from bench import build_workload
    from grapes_b200.dist import ShardedEmbedding, shard_batches
    from grapes_b200.engine import GrapesEngine
    from grapes_b200.graph import DeviceGraph
    world, rank = int(os.environ["WORLD_SIZE"]), int(os.environ["RANK"])
    dev = torch.device("cuda", int(os.environ["LOCAL_RANK"]))
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    cfg, indptr, indices, _x, y, train_idx = build_workload("products", 0, dev, native_csr=True)
    del _x
    N, B = cfg["N"], cfg["batch_size"]
    g = DeviceGraph(indptr, indices, N)
    table = torch.randn(N, 64, generator=torch.Generator().manual_seed(0))
    hp = dict(num_classes=cfg["C"], batch_size=B, num_samples=cfg["num_samples"], sampling_hops=cfg["sampling_hops"],
              embed_nodes=True, seed=rank)
    batches = [b.to(torch.int32).contiguous() for b in torch.split(train_idx, B)]
    batches = [batches[i] for i in shard_batches(len(batches), rank, world) if batches[i].numel() == B]
    res = {"rank": rank}
    for name in ("replicated", "sharded"):
        xin = ShardedEmbedding(table, dev) if name == "sharded" else table.to(dev)
        eng = GrapesEngine(g, xin, y, **hp)
        eng.enable_data_parallel(exchange="peer")
        for i in range(a.warmup):
            eng.step(batches[i % len(batches)], use_graph=True)
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(a.steps + 1)]
        ev[0].record()
        for i in range(a.steps):
            eng.step(batches[(a.warmup + i) % len(batches)], use_graph=True)
            ev[i + 1].record()
        torch.cuda.synchronize()
        eng.check_overflow()
        t = [ev[i].elapsed_time(ev[i + 1]) for i in range(a.steps)]
        held = (xin.table_bytes + xin.moment_bytes) if name == "sharded" else 3 * table.numel() * 4
        res[name] = {"ms_per_step_p50": pct(t, 50), "ms_per_step_p99": pct(t, 99), "table_and_moment_bytes": held,
                     "exchange": "peer" if eng.peer is not None else "nccl"}
        del eng, xin
        dist.barrier()
    outs = [None] * world
    dist.all_gather_object(outs, res)
    if rank == 0:
        with open(a.worker_out, "w") as f:
            json.dump(outs, f)
    dist.destroy_process_group()


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--out", required=True)
    p.add_argument("--shapes", default="products,papers")
    p.add_argument("--worlds", default="2,8")
    p.add_argument("--reps", type=int, default=20)
    p.add_argument("--rounds", type=int, default=7)
    p.add_argument("--steps", type=int, default=100)
    p.add_argument("--warmup", type=int, default=20)
    p.add_argument("--worker-out", dest="worker_out", default=None)
    a = p.parse_args()
    if a.worker_out:
        dp_worker(a)
        return
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_embed_sharded.py measures on a GPU; none is available")
    doc = {"what": "learned table (node_emb_dim 64) sharded by rows with its Adam moments vs replicated",
           **gpu_info()}
    doc["table_walk_1gpu"] = walk_bench(a)
    doc["engine_step_1gpu_products"] = engine_bench(a)
    doc["data_parallel"] = {}
    for w in (int(s) for s in a.worlds.split(",") if s):
        if torch.cuda.device_count() < w:
            doc["data_parallel"][f"W{w}"] = "not measured"
            continue
        with tempfile.TemporaryDirectory() as tmp:
            wout = os.path.join(tmp, "w.json")
            cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={w}",
                   "--master-addr", "127.0.0.1", "--master-port", "29563", os.path.abspath(__file__), "--out", a.out,
                   "--worker-out", wout, "--steps", str(a.steps), "--warmup", str(a.warmup)]
            r = subprocess.run(cmd, capture_output=True, text=True)
            doc["data_parallel"][f"W{w}"] = json.load(open(wout)) if r.returncode == 0 else \
                f"failed: {r.stdout[-1500:]} {r.stderr[-1500:]}"
    with open(a.out, "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps(doc))


if __name__ == "__main__":
    main()
