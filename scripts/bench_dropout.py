"""Cost of dropout in the classifier GCN (--dropout p): the training step with p = 0 against p = 0.5 on the products- and
arxiv-shaped synthetic graphs, both engines in one process on the same graph and batches, timed in alternating rounds.

    python scripts/bench_dropout.py --out result.json [--shapes products,arxiv] [--rounds 10] [--steps 20]

Per shape and p: ms/step of graph-replayed steps (CUDA events, p50 / p99 over all rounds), the launches of the step
graph, and the classifier part of the step alone (every launch tagged [cls]: the classifier's structure, forward, loss and
backward, each bracketed by CUDA events in eager steps, summed per step).  The GPU name and power limit are read in the
same run."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def pct(v, q):
    v = sorted(v)
    return v[min(len(v) - 1, int(round(q / 100.0 * (len(v) - 1))))]


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        info["nvidia_smi"] = [ln.strip() for ln in q.stdout.splitlines() if ln.strip()]
    except (OSError, subprocess.SubprocessError) as exc:
        info["nvidia_smi"] = f"not read: {exc}"
    return info


def run_shape(shape, a):
    import torch
    from bench import build_workload
    from grapes_b200.engine import GrapesEngine
    from grapes_b200.graph import DeviceGraph
    dev = torch.device("cuda", 0)
    cfg, indptr, indices, x, y, train_idx = build_workload(shape, 0, dev, native_csr=True)
    B = cfg["batch_size"]
    g = DeviceGraph(indptr, indices, cfg["N"])
    ps = (0.0, 0.5)
    engines = [GrapesEngine(g, x, y, num_classes=cfg["C"], batch_size=B, num_samples=cfg["num_samples"],
                            sampling_hops=cfg["sampling_hops"], seed=0, dropout=p) for p in ps]
    batches = [b.to(torch.int32).contiguous() for b in torch.split(train_idx, B) if b.numel() == B]
    seq = lambda i: batches[i % len(batches)]
    for e in engines:
        for i in range(a.warmup):
            e.step(seq(i), use_graph=True)
    torch.cuda.synchronize()
    step_ms = {p: [] for p in ps}
    for r in range(a.rounds):
        for p, e in zip(ps, engines):
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(a.steps + 1)]
            ev[0].record()
            for i in range(a.steps):
                e.step(seq(a.warmup + r * a.steps + i), use_graph=True)
                ev[i + 1].record()
            torch.cuda.synchronize()
            step_ms[p] += [ev[i].elapsed_time(ev[i + 1]) for i in range(a.steps)]
    for e in engines:
        e.check_overflow()
    # the classifier launches alone, event-bracketed in eager steps (profiling adds host work: a separate pass)
    cls_ms = {p: [] for p in ps}
    L = engines[0].L
    for r in range(a.cls_steps):
        for p, e in zip(ps, engines):
            L.profiling = True
            e.step(seq(r))
            summary = L.profile_summary()
            L.profiling = False
            cls_ms[p].append(sum(ms for name, (ms, _) in summary.items() if name.endswith("[cls]")))
    out = []
    for p, e in zip(ps, engines):
        out.append({"shape": shape, "dropout": p, "batch_size": B, "num_samples": cfg["num_samples"],
                    "sampling_hops": cfg["sampling_hops"], "cap_A": e.cap_A, "steps_timed": len(step_ms[p]),
                    "ms_per_step_p50": pct(step_ms[p], 50), "ms_per_step_p99": pct(step_ms[p], 99),
                    "classifier_ms_p50": pct(cls_ms[p], 50), "classifier_ms_p99": pct(cls_ms[p], 99),
                    "launches_per_graph": e.launches_per_graph,
                    "mask_bits_per_step": e.count("A") * (e.D + e.C) if p > 0 else 0})
    del engines, g
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="products,arxiv")
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--cls-steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_dropout.py measures on the GPU: no CUDA device")
    doc = {"bench": "dropout in the classifier GCN, p = 0 vs p = 0.5, alternating rounds in one process",
           **gpu_info(), "rounds": a.rounds, "steps_per_round": a.steps, "runs": []}
    for shape in a.shapes.split(","):
        for row in run_shape(shape, a):
            doc["runs"].append(row)
            print(json.dumps(row), flush=True)
    text = json.dumps(doc, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)
    print(text)


if __name__ == "__main__":
    main()
