"""Data-parallel training with a learned node-feature table (--embed_nodes, node_emb_dim = 64): time per step and the
cost of the step's tail (gradient exchange + parameter Adam + merge of the ranks' row-sparse table gradients + dense
table Adam), at 1, 2 and 8 ranks on the products- and arxiv-shaped synthetic graphs.

    python scripts/bench_embed_dp.py --out result.json [--worlds 1,2,8] [--shapes products,arxiv] [--steps 50]

The driver starts one ``torch.distributed.run`` per world size (world sizes above the box's GPU count are reported as not
measured) and prints / writes one JSON document with the GPU name and power limit read in the same run.  Per rank:
ms/step of graph-replayed steps (CUDA events, p50 / p99), target nodes/s, and the event-timed tail launches alone."""
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
    from grapes_b200.dist import shard_batches
    from grapes_b200.engine import GrapesEngine
    from grapes_b200.graph import DeviceGraph
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg, indptr, indices, _x, y, train_idx = build_workload(a.shape, 0, dev, native_csr=True)
    del _x
    N = cfg["N"]
    g = DeviceGraph(indptr, indices, N)
    gen = torch.Generator(device=dev).manual_seed(0)
    table = torch.randn(N, a.emb_dim, generator=gen, device=dev, dtype=torch.float32)
    B = cfg["batch_size"]
    eng = GrapesEngine(g, table, y, num_classes=cfg["C"], batch_size=B, num_samples=cfg["num_samples"],
                       sampling_hops=cfg["sampling_hops"], embed_nodes=True, seed=rank)
    if world > 1:
        eng.enable_data_parallel(exchange=a.exchange)
    exchange = "none" if world == 1 else ("peer" if eng.peer is not None else "nccl")
    batches = [b.to(torch.int32).contiguous() for b in torch.split(train_idx, B)]
    batches = [batches[i] for i in shard_batches(len(batches), rank, world) if batches[i].numel() == B]
    n = a.warmup + a.steps
    seq = [batches[i % len(batches)] for i in range(n)]
    for i in range(a.warmup):
        eng.step(seq[i], use_graph=True)
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(a.steps + 1)]
    ev[0].record()
    for i in range(a.steps):
        eng.step(seq[a.warmup + i], use_graph=True)
        ev[i + 1].record()
    torch.cuda.synchronize()
    eng.check_overflow()
    step_ms = [ev[i].elapsed_time(ev[i + 1]) for i in range(a.steps)]
    # the tail launches alone (grapes_step_tail[_embed] + grapes_embed_merge_adam, or grapes_adam_embed +
    # grapes_step_tail on one GPU) on the last step's gradients; every rank runs the same number of them, in lockstep
    st = torch.cuda.current_stream()
    tev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * a.tail_reps)]
    for i in range(a.tail_reps):
        tev[2 * i].record()
        eng._enqueue_tail(st.cuda_stream)
        tev[2 * i + 1].record()
    torch.cuda.synchronize()
    eng.check_overflow()
    tail_ms = [tev[2 * i].elapsed_time(tev[2 * i + 1]) for i in range(a.tail_reps)]
    A = eng.count("A")
    res = {"rank": rank, "exchange": exchange,
           "ms_per_step_p50": pct(step_ms, 50), "ms_per_step_p99": pct(step_ms, 99),
           "target_nodes_per_s_p50": B / (pct(step_ms, 50) / 1e3), "target_nodes_per_s_p99": B / (pct(step_ms, 99) / 1e3),
           "tail_ms_p50": pct(tail_ms, 50), "tail_ms_p99": pct(tail_ms, 99),
           "rows_last_step": A, "cap_A": eng.cap_A}
    rows = [res]
    if world > 1:
        rows = [None] * world
        dist.all_gather_object(rows, res)
    if rank == 0:
        F = a.emb_dim
        out = {"shape": a.shape, "world": world, "N": N, "node_emb_dim": F, "batch_size": B,
               "num_samples": cfg["num_samples"], "sampling_hops": cfg["sampling_hops"], "steps": a.steps,
               "warmup": a.warmup, "tail_reps": a.tail_reps,
               "payload_bytes_per_rank_max": eng.cap_A * (F + 1) * 4 + 16,
               "table_adam_bytes": 28 * N * F, "ranks": rows}
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
    ap.add_argument("--shapes", default="products,arxiv")
    ap.add_argument("--exchange", default="peer", choices=("peer", "nccl"))
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--tail-reps", type=int, default=30)
    ap.add_argument("--emb-dim", type=int, default=64)
    ap.add_argument("--out", default=None)
    ap.add_argument("--worker", action="store_true")
    ap.add_argument("--shape", default="products")
    ap.add_argument("--result", default=None)
    a = ap.parse_args()
    if a.worker:
        return worker(a)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_embed_dp.py measures on the GPU: no CUDA device")
    doc = {"bench": "data-parallel learned node features (embed_nodes)", "exchange": a.exchange, **gpu_info(), "runs": []}
    ngpu = torch.cuda.device_count()
    with tempfile.TemporaryDirectory() as tmp:
        for shape in a.shapes.split(","):
            for w in [int(v) for v in a.worlds.split(",")]:
                if w > ngpu:
                    doc["runs"].append({"shape": shape, "world": w, "result": f"not measured: {ngpu} GPUs on the box"})
                    continue
                res = os.path.join(tmp, f"{shape}_{w}.json")
                cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={w}",
                       "--master-addr", "127.0.0.1", "--master-port", str(29600 + w), os.path.abspath(__file__),
                       "--worker", "--shape", shape, "--result", res, "--exchange", a.exchange,
                       "--steps", str(a.steps), "--warmup", str(a.warmup), "--tail-reps", str(a.tail_reps),
                       "--emb-dim", str(a.emb_dim)]
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
