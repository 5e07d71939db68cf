"""Full-graph training (grapes_b200.full_batch) against the GRAPES epoch on the same graph, in one process.

For each synthetic shape (arxiv, Reddit, products by default): the one-off build of the gcn_norm structure in both
directions (canonical CSR, forward structure, transposed structure), then full-graph epochs of ``GCN(F, [256, C])`` --
forward + loss, backward + Adam -- event-timed after warm-up (p50), the peak allocated memory, and beside them the
GRAPES epoch: batches x the p50 step time of ``GrapesEngine`` (CUDA-graph replay, default configuration of the shape).
Writes one JSON object with the card name and power limit.

    python scripts/bench_full_batch.py --out /tmp/full_batch.json [--shapes arxiv,reddit,products] [--epochs 10]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        power = None
    return name, power


def _p50(xs):
    xs = sorted(xs)
    return xs[len(xs) // 2]


def bench_shape(shape, epochs, warmup, grapes_steps, dev):
    from grapes_b200 import full_batch as fb
    from grapes_b200.args import Arguments
    from grapes_b200.engine import GrapesEngine
    from grapes_b200.eval import WIDE_MIN_EDGES, _graph_norm
    from grapes_b200.graph import DeviceGraph
    from grapes_b200.synth import SHAPES, make_synth
    cfg = SHAPES[shape]
    d = make_synth(shape, seed=0, device=dev)
    args = Arguments(hidden_dim=256, seed=0)
    N, E = d.num_nodes, int(d.edge_index.shape[1])
    for _ in range(2):                    # the second build is timed: the first loads modules and warms the allocator
        graph = gn = None
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        graph = DeviceGraph.from_edge_index(d.edge_index, N, device=dev)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        gn = _graph_norm(graph, d, wide=E >= WIDE_MIN_EDGES)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        gn.build_transposed()
        torch.cuda.synchronize()
        t3 = time.perf_counter()

    gcn = fb.initial_model(args, d.num_features, d.num_classes).to(dev)
    opt = torch.optim.Adam(gcn.parameters(), lr=args.lr_gc)
    x, y, mask = d.x, d.y, d.train_mask
    torch.cuda.reset_peak_memory_stats(dev)
    fwd, bwd = [], []
    for i in range(warmup + epochs):
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record()
        logits, _ = gcn(x, gn)
        loss = fb.classifier_loss(logits, y, mask, 0.0)
        e[1].record()
        opt.zero_grad()
        loss.backward()
        opt.step()
        e[2].record()
        del logits, loss
        torch.cuda.synchronize()
        if i >= warmup:
            fwd.append(e[0].elapsed_time(e[1]))
            bwd.append(e[1].elapsed_time(e[2]))
    peak = torch.cuda.max_memory_allocated(dev)
    del gcn, opt
    graph._graph_norm = None
    del gn
    torch.cuda.empty_cache()

    # the GRAPES epoch on the same graph: batches x p50 step time
    B = cfg["batch_size"]
    eng = GrapesEngine(graph, x, y, num_classes=d.num_classes, batch_size=B, num_samples=cfg["num_samples"],
                       sampling_hops=cfg["sampling_hops"], hidden_dim=256, seed=0)
    train_idx = mask.nonzero().squeeze(1).to(torch.int32)
    nb = (train_idx.numel() + B - 1) // B
    batches = [train_idx[(j % nb) * B:((j % nb) + 1) * B].contiguous() for j in range(2 * grapes_steps)]
    for j in range(grapes_steps):                                   # warm-up: every graph variant captured
        eng.step(batches[j], use_graph=True)
    torch.cuda.synchronize()
    steps = []
    for j in range(grapes_steps, 2 * grapes_steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        eng.step(batches[j], use_graph=True)
        b.record()
        steps.append((a, b))
    torch.cuda.synchronize()
    eng.check_overflow()
    step_ms = _p50([a.elapsed_time(b) for a, b in steps])
    del eng
    return {
        "N": N, "E": E, "F": d.num_features, "C": d.num_classes, "hidden": 256,
        "structure": "GraphNorm" if E < WIDE_MIN_EDGES else "WideGraphNorm",
        "build_ms": {"csr": 1e3 * (t1 - t0), "forward_structure": 1e3 * (t2 - t1), "transposed_structure": 1e3 * (t3 - t2)},
        "epoch_ms_p50": _p50([f + b for f, b in zip(fwd, bwd)]),
        "forward_ms_p50": _p50(fwd), "backward_adam_ms_p50": _p50(bwd),
        "epochs_timed": epochs, "warmup_epochs": warmup,
        "peak_allocated_bytes": int(peak),
        "grapes": {"batches_per_epoch": nb, "batch_size": B, "step_ms_p50": step_ms, "steps_timed": grapes_steps,
                   "epoch_ms": nb * step_ms},
    }


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--shapes", default="arxiv,reddit,products")
    ap.add_argument("--epochs", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--grapes-steps", type=int, default=50)
    a = ap.parse_args(argv)
    if not torch.cuda.is_available():
        print("bench_full_batch.py: no CUDA device -- grapes_b200 has no CPU fallback", file=sys.stderr)
        return 2
    dev = torch.device("cuda", 0)
    name, power = _card()
    out = {"card": name, "power_limit": power, "shapes": {}}
    for shape in a.shapes.split(","):
        out["shapes"][shape] = bench_shape(shape, a.epochs, a.warmup, a.grapes_steps, dev)
        print(shape, json.dumps(out["shapes"][shape]), flush=True)
        torch.cuda.empty_cache()
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))
    return 0


if __name__ == "__main__":
    sys.exit(main())
