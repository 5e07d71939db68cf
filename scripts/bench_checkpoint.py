"""Save and load time of a checkpoint (grapes_b200.checkpoint) on the products shape with learned node features
(--embed_nodes, F = 64: the table and its two Adam moments are 3 x 627 MB, the parameters and their moments under 2 MB).

    python scripts/bench_checkpoint.py --out result.json [--reps 3] [--dir DIR]

Measured, each --reps times (median and all values):
  * save() of the replicated engine (every file written, fsynced, committed) and load() back into it;
  * the same for an engine over an emulated W = 8 sharded table (one process writes and reads all eight shards);
  * one W = 8 shard alone: write_rows() of its rows of the three table files, and ShardedEmbedding.load_rows() of them --
    what one rank of an 8-GPU box moves.
Bytes, seconds and GB/s are reported.  The load follows the save at once, so its reads come from the page cache; the
saves end in fsync, so they include the device.  The GPU name, its power limit and the filesystem of the checkpoint
directory are read in the same run."""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    import torch
    out = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        out["power_limit_and_max_sm_clock"] = q[0] if q else "unknown"
    except Exception as exc:                           # noqa: BLE001
        out["power_limit_and_max_sm_clock"] = f"unknown ({exc})"
    return out


def filesystem(path):
    """(mount point, type, device) of the mount that holds ``path``, from /proc/mounts."""
    path = os.path.realpath(path)
    best = ("", "unknown", "unknown")
    try:
        with open("/proc/mounts") as f:
            for ln in f:
                dev, mnt, typ = ln.split()[:3]
                inside = path == mnt or path.startswith(mnt.rstrip("/") + "/")
                if inside and len(mnt) >= len(best[0]):
                    best = (mnt, typ, dev)
    except OSError:
        pass
    return dict(mount=best[0], type=best[1], device=best[2])


def timed(fn, reps):
    import torch
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return ts


def line(name, nbytes, ts):
    med = sorted(ts)[len(ts) // 2]
    return dict(what=name, bytes=int(nbytes), seconds_median=med, seconds_all=ts, gb_per_s=nbytes / med / 1e9)


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--out", required=True)
    p.add_argument("--reps", type=int, default=3)
    p.add_argument("--dir", default=None, help="checkpoint directory parent (default: a temporary directory)")
    a = p.parse_args()
    import torch
    from grapes_b200 import checkpoint as C
    from grapes_b200.dist import ShardedEmbedding, feature_bounds
    from grapes_b200.engine import GrapesEngine
    from grapes_b200.graph import DeviceGraph
    from grapes_b200.synth import SHAPES, make_synth
    if not torch.cuda.is_available():
        raise SystemExit("bench_checkpoint.py measures on a GPU; none is visible")
    dev = torch.device("cuda:0")
    cfg = SHAPES["products"]
    F, W = 64, 8
    d = make_synth("products", seed=0, device=dev, features=False)
    g = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=dev)
    del d.edge_index
    N = d.num_nodes
    table = torch.empty(N, F, device=dev).normal_(generator=torch.Generator(device=dev).manual_seed(1))
    idx = d.train_mask.nonzero().squeeze(1).to(torch.int32)
    batches = [b.contiguous() for b in torch.split(idx, cfg["batch_size"])][:3]
    base = a.dir or tempfile.mkdtemp(prefix="grapes_ckpt_bench_")
    os.makedirs(base, exist_ok=True)
    out = dict(gpu_info(), filesystem=filesystem(base), shape="products", N=N, F=F, reps=a.reps, lines=[])

    def engine(x):
        e = GrapesEngine(g, x, d.y, num_classes=d.num_classes, batch_size=cfg["batch_size"],
                         num_samples=cfg["num_samples"], sampling_hops=cfg["sampling_hops"], hidden_dim=256, seed=0,
                         embed_nodes=True)
        for b in batches:                              # non-zero moments, a real step count
            e.step(b)
        torch.cuda.synchronize()
        e.check_overflow()
        return e

    try:
        for name, x in (("replicated", table.clone()), (f"emulated W={W}", ShardedEmbedding.emulate(table, W)[W - 1])):
            e = engine(x)
            ck = os.path.join(base, name.replace(" ", "_").replace("=", ""))
            step = [0]

            def save():
                step[0] += 1
                C.save(e, ck, dict(step=step[0]))
            ts = timed(save, a.reps)
            path = C.latest(ck)
            nbytes = sum(os.path.getsize(os.path.join(path, f)) for f in os.listdir(path))
            out["lines"].append(line(f"save, {name}", nbytes, ts))
            out["lines"].append(line(f"load, {name}", nbytes, timed(lambda: C.load(e, path), a.reps)))
            if name.startswith("emulated"):
                s = e.embed_shards.shards[0]
                n = s.hi - s.lo
                one = os.path.join(base, "one_shard")
                os.makedirs(one, exist_ok=True)

                def write_one():
                    for f, t in zip(C.TABLE_FILES, (s.table.rows[:n, :F], s.exp_avg[:n], s.exp_avg_sq[:n])):
                        C.write_rows(os.path.join(one, f), t, s.lo, N)
                ts = timed(write_one, a.reps)
                sb = 3 * n * F * 4
                out["lines"].append(line(f"write_rows, one shard of W={W} (rows {s.lo}..{s.hi})", sb, ts))
                src = C.table_source(path)
                out["lines"].append(line(f"load_rows, one shard of W={W}", sb, timed(lambda: s.load_rows(*src), a.reps)))
                out["papers_per_rank_bytes_W8_arithmetic"] = 3 * (feature_bounds(111_059_956, W)[1]) * F * 4
            del e
            torch.cuda.empty_cache()
    finally:
        if a.dir is None:
            shutil.rmtree(base, ignore_errors=True)
    for ln in out["lines"]:
        print(f"{ln['what']:<52} {ln['bytes'] / 1e6:10.1f} MB  {ln['seconds_median']:8.3f} s  {ln['gb_per_s']:6.2f} GB/s",
              flush=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
