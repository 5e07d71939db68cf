"""torchrun --nproc-per-node 2 scripts/check_dp_eval.py
Data-parallel evaluation (``eval.evaluate(..., group=...)``) against one process on the same weights:
  1. full batch: every rank's (accuracy, f1) equals the one-process evaluate(); each rank's window logits equal the same
     rows of the one-process logits bit for bit (layer 2 read Z over peer memory);
  2. mini batch: the same scores, and return_predictions gives the one-process tensor on every rank;
  3. a peer-mapping failure forced on one rank, and a classifier the row-slab forward does not cover (D <= C), send
     every rank to the replicated evaluation with the same scores;
  4. train() with shard_eval=True and shard_eval=False returns the same test_f1 and logs the same lines, full batch and
     mini batch.
Prints "dp eval ok" on rank 0."""
import logging
import os
import sys
import warnings

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import grapes_b200.dist as D                                     # noqa: E402
from grapes_b200 import eval as E                                # noqa: E402
from grapes_b200.gcn import GCN, full_graph_forward_sharded      # noqa: E402
from grapes_b200.graph import DeviceGraph                        # noqa: E402
from grapes_b200.synth import SHAPES, make_synth                 # noqa: E402


def setup(name, dev, seed=0, multilabel=False):
    cfg = SHAPES[name]
    d = make_synth(name, seed=seed, multilabel=multilabel)
    torch.manual_seed(seed)                                      # the same weights on every rank
    gcn_c = GCN(d.num_features, [256, d.num_classes]).to(dev).eval()
    gcn_gf = GCN(d.num_features + cfg["sampling_hops"] + 1, [256, 1]).to(dev)      # + the hop indicators
    args = type("A", (), dict(sampling_hops=cfg["sampling_hops"], num_samples=cfg["num_samples"], use_indicators=True,
                              batch_size=cfg["batch_size"]))()
    return d, gcn_c, gcn_gf, args


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = torch.device("cuda", int(os.environ["LOCAL_RANK"]))
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    G = dist.group.WORLD
    for name, ml in (("small", False), ("cora", False), ("tiny", True)):
        d, gcn_c, gcn_gf, args = setup(name, dev, multilabel=ml)
        nind = args.sampling_hops + 1
        mask = d.val_mask if ml else d.test_mask
        g = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=dev)
        one = E.evaluate(gcn_c, gcn_gf, d, args, g, None, nind, dev, mask=mask, full_batch=True, return_predictions=True)
        dp = E.evaluate(gcn_c, gcn_gf, d, args, g, None, nind, dev, mask=mask, full_batch=True, group=G)
        assert dp == one[:2], (name, dp, one[:2])
        _, sgn, table = g._sharded_eval
        assert table is not None, "peer row table was not set up"
        lg, _ = full_graph_forward_sharded(gcn_c, d.x.to(dev), sgn, table, return_logits=True)
        assert torch.equal(lg, one[2][sgn.lo:sgn.hi]), f"{name}: window logits of rank {rank} differ"
        if not ml:
            idx = mask.nonzero().squeeze(1)
            loader = [(b,) for b in torch.split(idx, args.batch_size)]
            one_mb = E.evaluate(gcn_c, gcn_gf, d, args, g, None, nind, dev, mask=mask, loader=loader, full_batch=False,
                                return_predictions=True)
            dp_mb = E.evaluate(gcn_c, gcn_gf, d, args, g, None, nind, dev, mask=mask, loader=loader, full_batch=False,
                               return_predictions=True, group=G)
            assert dp_mb[:2] == one_mb[:2], (name, dp_mb[:2], one_mb[:2])
            assert torch.equal(dp_mb[2], one_mb[2])
        print(f"rank {rank} {name}: full {dp} window rows {sgn.rows}", flush=True)

    # forced mapping failure on rank 1
    d, gcn_c, gcn_gf, args = setup("small", dev)
    nind = args.sampling_hops + 1
    g = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=dev)
    one = E.evaluate(gcn_c, gcn_gf, d, args, g, None, nind, dev, mask=d.test_mask, full_batch=True)
    real = D.PeerRowTable.__init__

    def failing(self, *a, **kw):
        if dist.get_rank() == 1:
            raise RuntimeError("forced mapping failure")
        real(self, *a, **kw)
    D.PeerRowTable.__init__ = failing
    try:
        with warnings.catch_warnings(record=True) as caught:
            warnings.simplefilter("always")
            res = E.evaluate(gcn_c, gcn_gf, d, args, g, None, nind, dev, mask=d.test_mask, full_batch=True, group=G)
    finally:
        D.PeerRowTable.__init__ = real
    assert res == one, (res, one)
    assert g._sharded_eval[2] is None and any("replicated" in str(w.message) for w in caught)

    # a classifier the row-slab forward does not cover (hidden width D <= C): every rank evaluates replicated
    d = make_synth("small", seed=3)
    torch.manual_seed(3)
    narrow = GCN(d.num_features, [d.num_classes - 1, d.num_classes]).to(dev).eval()
    g = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=dev)
    one = E.evaluate(narrow, gcn_gf, d, args, g, None, nind, dev, mask=d.test_mask, full_batch=True)
    res = E.evaluate(narrow, gcn_gf, d, args, g, None, nind, dev, mask=d.test_mask, full_batch=True, group=G)
    assert res == one and getattr(g, "_sharded_eval", None) is None, (res, one)

    # train(): sharded and replicated evaluation, same results and logs
    from grapes_b200 import train as T
    from grapes_b200.args import Arguments
    for full in (True, False):
        runs = []
        for shard in (True, False):
            lines = []
            log = logging.getLogger("check_dp_eval")
            log.handlers, log.propagate = [], False
            h = logging.Handler()
            h.emit = lambda rec: lines.append(rec.getMessage())
            log.addHandler(h)
            log.setLevel("INFO")
            T.get_logger = lambda: log
            a = Arguments()
            a.dataset, a.max_epochs, a.batch_size, a.num_samples, a.sampling_hops = "small", 2, 128, 32, 3
            a.eval_frequency, a.eval_full_batch = 1, full
            f1, *_ = T.train(a, data=make_synth("small", seed=2), device=dev, shard_eval=shard)
            runs.append((f1, lines))
        assert runs[0] == runs[1], (full, runs)
        print(f"rank {rank} train full_batch={full}: test_f1 {runs[0][0]}, {len(runs[0][1])} log lines", flush=True)
    dist.barrier()
    if rank == 0:
        print(f"dp eval ok: world={world}", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    try:
        main()
    except BaseException:
        import traceback
        print("RANK", os.environ.get("RANK"), "FAILED:\n" + traceback.format_exc(), flush=True)
        raise
