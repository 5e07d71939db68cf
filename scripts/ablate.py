"""Timing experiments on the products-shaped workload: the step graph with parts left out
(`GrapesEngine.ablate`) or on one stream, to see what sits on the critical path.
Not a benchmark: results of ablated steps are wrong by construction."""
import os, sys, json, time
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import build_workload
from grapes_b200.engine import GrapesEngine
from grapes_b200.graph import DeviceGraph

PREFETCH = os.environ.get("GRAPES_NO_PREFETCH") is None


def main():
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    cfg, indptr, indices, x, y, train_idx = build_workload(sys.argv[1] if len(sys.argv) > 1 else "products", 0, dev)
    N, F, C, B = cfg["N"], cfg["F"], cfg["C"], cfg["batch_size"]
    graph = DeviceGraph(indptr, indices, N)
    nb = train_idx.numel() // B
    batches = torch.stack([train_idx[b * B:(b + 1) * B] for b in range(41)]).to(torch.int32)
    variants = [("full", {}, ""), ("one_stream", dict(multi_stream=False), ""), ("nobwd", {}, "nobwd"),
                ("nocls", {}, "nocls"), ("nobwd_nocls", {}, "nobwd,nocls")]
    out = {}
    for name, kw, abl in variants:
        eng = GrapesEngine(graph, x, y, num_classes=C, batch_size=B, num_samples=cfg["num_samples"],
                           sampling_hops=cfg["sampling_hops"], hidden_dim=256, seed=0, **kw)
        eng.ablate = set(filter(None, abl.split(",")))
        for j in range(5):
            eng.step(batches[j], use_graph=True, next_targets=batches[j + 1] if PREFETCH else None)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for j in range(5, 35):
            eng.step(batches[j], use_graph=True, next_targets=batches[j + 1] if PREFETCH else None)
        e1.record(); torch.cuda.synchronize()
        out[name] = round(e0.elapsed_time(e1) / 30, 4)
        del eng
    print(json.dumps(out))

if __name__ == "__main__":
    main()
