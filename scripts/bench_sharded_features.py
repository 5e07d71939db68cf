"""A feature table sharded across the data-parallel ranks against the replicated table: time per training step (p50 /
p99), per-rank device memory of the table, and the feature bytes each step reads from other ranks' shards, on the
products- and papers-shaped synthetic graphs.

    python scripts/bench_sharded_features.py --out result.json [--worlds 1,2,8] [--shapes products,papers] [--steps 60]

The driver starts one ``torch.distributed.run`` per world size (world sizes above the box's GPU count are reported as not
measured) and writes one JSON document with the GPU name and power limit read in the same run.  Each rank builds a
replicated engine and one over ``ShardedFeatures`` (same seed, same batches) and times them in alternating rounds of
``--round`` graph-replayed steps (CUDA events).  World 1 is a one-GPU stand-in: the table is split into ``--emulate``
allocations of the one device, which measures the register-staged peer gather against the replicated (TMA-staged) one
without any NVLink traffic.  Remote bytes per step are computed from the recorded sizes of the last step: every hop reads
n + nnz feature rows and the classifier A + nnz, each row from another rank with probability 1 - 1/W (uniform ids)."""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def pct(v, q):
    v = sorted(v)
    return v[min(len(v) - 1, int(round(q / 100.0 * (len(v) - 1))))]


def worker(a):
    import torch
    import torch.distributed as dist
    from bench import build_workload
    from grapes_b200.dist import ShardedFeatures, shard_batches
    from grapes_b200.engine import GrapesEngine
    from grapes_b200.graph import DeviceGraph
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg, indptr, indices, x, y, train_idx = build_workload(a.shape, 0, dev, native_csr=True)
    N, B = cfg["N"], cfg["batch_size"]
    g = DeviceGraph(indptr, indices, N)
    m0 = torch.cuda.memory_allocated(dev)
    feats = ShardedFeatures(x, dev) if world > 1 else ShardedFeatures.emulate(x, a.emulate)[0]
    shard_mem = torch.cuda.memory_allocated(dev) - m0
    W = feats.world
    kw = dict(num_classes=cfg["C"], batch_size=B, num_samples=cfg["num_samples"], sampling_hops=cfg["sampling_hops"],
              seed=rank)
    engines = {"replicated": GrapesEngine(g, x, y, **kw), "sharded": GrapesEngine(g, feats, y, **kw)}
    batches = [b.to(torch.int32).contiguous() for b in torch.split(train_idx, B)]
    batches = [batches[i] for i in shard_batches(len(batches), rank, world) if batches[i].numel() == B]
    times = {k: [] for k in engines}
    for k, eng in engines.items():
        for i in range(a.warmup):
            eng.step(batches[i % len(batches)], use_graph=True)
    torch.cuda.synchronize()
    done = 0
    while done < a.steps:
        n = min(a.round, a.steps - done)
        for k, eng in engines.items():
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(n + 1)]
            ev[0].record()
            for i in range(n):
                eng.step(batches[(done + i) % len(batches)], use_graph=True)
                ev[i + 1].record()
            torch.cuda.synchronize()
            times[k] += [ev[i].elapsed_time(ev[i + 1]) for i in range(n)]
        done += n
    rows_read = 0
    for eng in engines.values():
        eng.check_overflow()
    eng = engines["sharded"]
    for h in eng.hop_sizes():
        rows_read += h["n"] + h["nnz"]
    rows_read += eng.count("A") + eng.count("cl_nnz")
    row_bytes = cfg["F"] * x.element_size()
    res = {"rank": rank, "table_device_bytes_sharded": shard_mem, "table_device_bytes_replicated": x.numel() * x.element_size(),
           "feature_rows_read_last_step": rows_read,
           "remote_feature_bytes_last_step": int(rows_read * row_bytes * (1 - 1 / W)) if world > 1 else 0}
    for k, v in times.items():
        res[f"{k}_ms_p50"], res[f"{k}_ms_p99"] = pct(v, 50), pct(v, 99)
    rows = [res]
    if world > 1:
        rows = [None] * world
        dist.all_gather_object(rows, res)
    if rank == 0:
        out = {"shape": a.shape, "world": world, "shards": W, "N": N, "F": cfg["F"],
               "feature_dtype": str(x.dtype).replace("torch.", ""), "batch_size": B, "steps": a.steps,
               "warmup": a.warmup, "round": a.round, "ranks": rows}
        with open(a.result, "w") as f:
            json.dump(out, f)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0), "gpus_on_box": torch.cuda.device_count()}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        info["nvidia_smi"] = [ln.strip() for ln in q.stdout.splitlines() if ln.strip()]
    except (OSError, subprocess.SubprocessError) as exc:
        info["nvidia_smi"] = f"not read: {exc}"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--worlds", default="1,2,8")
    ap.add_argument("--shapes", default="products,papers")
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--round", type=int, default=10)
    ap.add_argument("--emulate", type=int, default=8)
    ap.add_argument("--out", default=None)
    ap.add_argument("--worker", action="store_true")
    ap.add_argument("--shape", default="products")
    ap.add_argument("--result", default=None)
    a = ap.parse_args()
    if a.worker:
        return worker(a)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_sharded_features.py measures on the GPU: no CUDA device")
    doc = {"bench": "feature table sharded across the data-parallel ranks vs replicated", **gpu_info(), "runs": []}
    ngpu = torch.cuda.device_count()
    with tempfile.TemporaryDirectory() as tmp:
        for shape in a.shapes.split(","):
            for w in [int(v) for v in a.worlds.split(",")]:
                if w > ngpu:
                    doc["runs"].append({"shape": shape, "world": w, "result": f"not measured: {ngpu} GPUs on the box"})
                    continue
                res = os.path.join(tmp, f"{shape}_{w}.json")
                cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={w}",
                       "--master-addr", "127.0.0.1", "--master-port", str(29700 + w), os.path.abspath(__file__),
                       "--worker", "--shape", shape, "--result", res, "--steps", str(a.steps),
                       "--warmup", str(a.warmup), "--round", str(a.round), "--emulate", str(a.emulate)]
                p = subprocess.run(cmd, capture_output=True, text=True, timeout=1800)
                if p.returncode != 0 or not os.path.isfile(res):
                    doc["runs"].append({"shape": shape, "world": w, "result": "failed",
                                        "log": (p.stdout[-3000:] + p.stderr[-3000:])})
                    continue
                with open(res) as f:
                    doc["runs"].append(json.load(f))
                print(json.dumps(doc["runs"][-1]), flush=True)
    text = json.dumps(doc, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)
    print(text)


if __name__ == "__main__":
    main()
