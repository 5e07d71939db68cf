"""Data-parallel full-graph training (grapes_b200.full_batch.WindowEpoch) on one B200, products shape by default.

1. The W = 1 data-parallel epoch (one window holding every row: forward, window loss, backward over the transposed
   window, rank-order sum, Adam) against the one-GPU epoch of the drop-in module (``gcn(x, GraphNorm)`` + main.py's loss
   + backward + Adam), alternated epoch by epoch, p50 over ``--epochs`` after ``--warmup`` warm-up epochs each.
2. The per-rank phase times of an EMULATED W = 8 run: the eight windows' phases run one after another on this one
   device, with row tables in local memory.  No NVLink traffic, no concurrency: these are the work of each rank's share,
   not an 8-GPU epoch time; multi-GPU speed-up is not measured here.
Writes one JSON object with the card name and power limit read in the same run.

    python scripts/bench_full_batch_dp.py --out /tmp/full_batch_dp.json [--shape products] [--epochs 10] [--warmup 3]
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
from bench_full_batch import _card, _p50                           # noqa: E402


def _windows(graph, d, W, C4, D, dev):
    from grapes_b200.full_batch import WindowEpoch
    from grapes_b200.gcn import LocalRowTable, ShardedGraphNorm
    sgns = [ShardedGraphNorm(graph, W, r, edge_index=d.edge_index) for r in range(W)]
    rows = max(s.rows for s in sgns)
    zt = LocalRowTable.make(W, rows, C4, dev)
    dt = LocalRowTable.make(W, rows, D, dev) if d.num_features > D else [None] * W
    for s in sgns:
        s.build_transposed()
    return sgns, zt, dt


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--shape", default="products")
    ap.add_argument("--epochs", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--world", type=int, default=8)
    a = ap.parse_args(argv)
    if not torch.cuda.is_available():
        print("bench_full_batch_dp.py: no CUDA device -- grapes_b200 has no CPU fallback", file=sys.stderr)
        return 2
    from grapes_b200 import full_batch as fb
    from grapes_b200.args import Arguments
    from grapes_b200.eval import _graph_norm
    from grapes_b200.graph import DeviceGraph
    from grapes_b200.synth import make_synth
    dev = torch.device("cuda", 0)
    name, power = _card()
    d = make_synth(a.shape, seed=0, device=dev)
    args = Arguments(hidden_dim=256, seed=0)
    D, C = 256, d.num_classes
    C4 = (C + 3) // 4 * 4
    x, y, mask = d.x, d.y, d.train_mask
    n_train = int(mask.sum())
    graph = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=dev)
    gn = _graph_norm(graph, d)
    gn.build_transposed()

    one = fb.initial_model(args, d.num_features, C).to(dev)
    opt_one = torch.optim.Adam(one.parameters(), lr=args.lr_gc)
    dp = fb.initial_model(args, d.num_features, C).to(dev)
    opt_dp = torch.optim.Adam(dp.parameters(), lr=args.lr_gc)
    sgns, zt, dt = _windows(graph, d, 1, C4, D, dev)
    ep = fb.WindowEpoch(dp, x, sgns[0], zt[0], y, mask, n_train, 0.0, dt[0])

    def one_gpu_epoch():
        logits, _ = one(x, gn)
        loss = fb.classifier_loss(logits, y, mask, 0.0)
        opt_one.zero_grad()
        loss.backward()
        opt_one.step()

    def dp_epoch():
        fb._set_grads(dp, fb.run_epoch_emulated([ep]))
        opt_dp.step()

    times = {"one_gpu": [], "dp_w1": []}
    for i in range(a.warmup + a.epochs):
        for key, fn in (("one_gpu", one_gpu_epoch), ("dp_w1", dp_epoch)):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            if i >= a.warmup:
                times[key].append(e0.elapsed_time(e1))
    # the first epoch of both starts from the same weights: their forward logits agree bit for bit (checked once here)
    same = {n: p.detach().clone() for n, p in fb.initial_model(args, d.num_features, C).named_parameters()}
    for m in (one, dp):
        m.load_state_dict(same)
    with torch.no_grad():
        ref, _ = one(x, gn)
    ep.phases()[0]()
    ep.phases()[1]()
    logits_equal = bool(torch.equal(ep.logits, ref))
    del ref, ep, sgns, zt, dt, opt_one, one
    graph._graph_norm = None
    del gn
    torch.cuda.empty_cache()

    # emulated W ranks: every rank's phase k, one after another, each event-timed
    W = a.world
    sgns, zt, dt = _windows(graph, d, W, C4, D, dev)
    eps = [fb.WindowEpoch(dp, x, s, z, y, mask, n_train, 0.0, t) for s, z, t in zip(sgns, zt, dt)]
    nph = len(eps[0].phases())
    per = [[[] for _ in range(nph)] for _ in range(W)]
    for i in range(a.warmup + a.epochs):
        for k in range(nph):
            for r, e in enumerate(eps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                e.phases()[k]()
                e1.record()
                torch.cuda.synchronize()
                if i >= a.warmup:
                    per[r][k].append(e0.elapsed_time(e1))
        fb._set_grads(dp, fb.sum_in_rank_order([e.partial() for e in eps]))
        opt_dp.step()
    phase_ms = [[_p50(per[r][k]) for k in range(nph)] for r in range(W)]
    rank_ms = [sum(p) for p in phase_ms]
    out = {
        "card": name, "power_limit": power, "shape": a.shape,
        "N": d.num_nodes, "E": int(d.edge_index.shape[1]), "F": d.num_features, "C": C, "hidden": D,
        "epochs_timed": a.epochs, "warmup_epochs": a.warmup,
        "w1_vs_one_gpu": {
            "order": "alternated epoch by epoch, one-GPU first",
            "one_gpu_epoch_ms_p50": _p50(times["one_gpu"]), "dp_w1_epoch_ms_p50": _p50(times["dp_w1"]),
            "one_gpu_epoch_ms": times["one_gpu"], "dp_w1_epoch_ms": times["dp_w1"],
            "first_epoch_logits_bit_identical": logits_equal,
        },
        f"emulated_w{W}": {
            "note": (f"one-device emulation of {W} ranks without NVLink traffic: each rank's phases run one after "
                     f"another on this GPU; not an {W}-GPU epoch time"),
            "phases": ["layer1", "layer2_loss", "publish_dlogits", "backward2"] + (["backward1"] if nph == 5 else []),
            "window_rows": [s.rows for s in sgns],
            "phase_ms_p50": phase_ms, "rank_ms": rank_ms, "max_rank_ms": max(rank_ms),
            "max_phase_ms": [max(phase_ms[r][k] for r in range(W)) for k in range(nph)],
        },
    }
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))
    return 0


if __name__ == "__main__":
    sys.exit(main())
