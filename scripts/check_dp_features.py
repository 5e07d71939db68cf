"""torchrun --nproc-per-node 2 scripts/check_dp_features.py
A feature table sharded across the ranks (``dist.ShardedFeatures`` over real symmetric memory) against the replicated
table:
  1. each rank's shard holds rows bounds[r] .. bounds[r + 1] of the table and about 1/W of its bytes;
  2. full-batch evaluation over the sharded table (F <= D and F > D) and mini-batch evaluation give the scores of the
     replicated one-process evaluate();
  3. train(shard_features=True) and train(shard_features=False) give bit-identical parameters and the same test_f1 and
     log lines, full batch and mini batch;
  4. a Python-level allocation failure injected on rank 1 makes every rank raise GrapesError.
Prints "dp features ok" on rank 0."""
import logging
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import grapes_b200.dist as D                                     # noqa: E402
from grapes_b200 import eval as E                                # noqa: E402
from grapes_b200._lib import GrapesError                         # noqa: E402
from grapes_b200.gcn import GCN                                  # noqa: E402
from grapes_b200.graph import DeviceGraph                        # noqa: E402
from grapes_b200.synth import SHAPES, make_synth                 # noqa: E402


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = torch.device("cuda", int(os.environ["LOCAL_RANK"]))
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    G = dist.group.WORLD
    for name, bf16 in (("small", False), ("small", True), ("cora", False)):
        cfg = SHAPES[name]
        d = make_synth(name, seed=1)
        if bf16:
            d.x = d.x.bfloat16()
        feats = D.ShardedFeatures(d.x, dev)                      # d.x stays on the host
        lo, hi = feats.bounds[rank], feats.bounds[rank + 1]
        assert torch.equal(feats.local.cpu(), d.x[lo:hi]), "shard rows differ from the table"
        whole = d.x.shape[0] * feats.ldx * d.x.element_size()
        assert feats.table_bytes <= whole / world + feats.ldx * d.x.element_size() * world, (feats.table_bytes, whole)
        torch.manual_seed(0)
        gcn_c = GCN(d.num_features, [256, d.num_classes]).to(dev).eval()
        gcn_gf = GCN(d.num_features + cfg["sampling_hops"] + 1, [256, 1]).to(dev)
        args = type("A", (), dict(sampling_hops=cfg["sampling_hops"], num_samples=cfg["num_samples"],
                                  use_indicators=True, batch_size=cfg["batch_size"]))()
        nind = cfg["sampling_hops"] + 1
        g = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=dev)
        one = E.evaluate(gcn_c, gcn_gf, d, args, g, None, nind, dev, mask=d.test_mask, full_batch=True)
        got = E.evaluate(gcn_c, gcn_gf, d, args, g, None, nind, dev, mask=d.test_mask, full_batch=True, group=G,
                         features=feats)
        assert got == one, (name, bf16, got, one)
        idx = d.test_mask.nonzero().squeeze(1)
        loader = [(b,) for b in torch.split(idx, cfg["batch_size"])]
        one_mb = E.evaluate(gcn_c, gcn_gf, d, args, g, None, nind, dev, mask=d.test_mask, loader=loader,
                            full_batch=False)
        got_mb = E.evaluate(gcn_c, gcn_gf, d, args, g, None, nind, dev, mask=d.test_mask, loader=loader,
                            full_batch=False, group=G, features=feats)
        assert got_mb == one_mb, (name, bf16, got_mb, one_mb)
        print(f"rank {rank} {name} bf16={bf16}: shard {feats.table_bytes} of {whole} bytes, full {got}, "
              f"mini-batch {got_mb}", flush=True)

    # train(): sharded and replicated tables, same parameters, scores and logs
    from grapes_b200 import train as T
    from grapes_b200.args import Arguments
    for full in (True, False):
        runs = []
        for shard in (True, False):
            lines = []
            log = logging.getLogger("check_dp_features")
            log.handlers, log.propagate = [], False
            h = logging.Handler()
            h.emit = lambda rec: lines.append(rec.getMessage())
            log.addHandler(h)
            log.setLevel("INFO")
            T.get_logger = lambda: log
            a = Arguments()
            a.dataset, a.max_epochs, a.batch_size, a.num_samples, a.sampling_hops = "small", 2, 128, 32, 3
            a.eval_frequency, a.eval_full_batch = 1, full
            f1, *_ = T.train(a, data=make_synth("small", seed=2), device=dev, shard_features=shard)
            eng = T.train.last_engine
            assert (eng.features is not None) == shard
            runs.append((f1, lines, eng.params.clone()))
        assert runs[0][:2] == runs[1][:2], (full, runs[0][:2], runs[1][:2])
        assert torch.equal(runs[0][2], runs[1][2]), "parameters differ between sharded and replicated tables"
        print(f"rank {rank} train full_batch={full}: test_f1 {runs[0][0]}, {len(runs[0][1])} log lines", flush=True)

    # an allocation failure on rank 1: every rank raises
    real = D.PeerRowTable.__init__

    def failing(self, *a, **kw):
        if dist.get_rank() == 1:
            raise RuntimeError("injected allocation failure")
        real(self, *a, **kw)
    D.PeerRowTable.__init__ = failing
    try:
        D.ShardedFeatures(make_synth("tiny", seed=0).x, dev)
        raise AssertionError("ShardedFeatures did not raise")
    except GrapesError as exc:
        assert ("this rank" in str(exc)) == (rank == 1), str(exc)
    finally:
        D.PeerRowTable.__init__ = real
    dist.barrier()
    if rank == 0:
        print(f"dp features ok: world={world}", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    try:
        main()
    except BaseException:
        import traceback
        print("RANK", os.environ.get("RANK"), "FAILED:\n" + traceback.format_exc(), flush=True)
        raise
