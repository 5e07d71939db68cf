"""``evaluate(..., group=...)`` with two processes on ONE B200 and a gloo group: the parts of the data-parallel evaluation
that need no peer memory.  A classifier the row-slab forward does not cover (hidden width D <= C) falls back to the
replicated full-batch evaluation on every rank with the one-process scores; mini-batch evaluation splits the batches
between the ranks and returns the one-process scores and predictions."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from grapes_b200 import eval as E
    from grapes_b200.gcn import GCN
    from grapes_b200.graph import DeviceGraph
    from grapes_b200.synth import SHAPES, make_synth
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    G = dist.group.WORLD
    res = {}
    for name in ("small", "cora"):
        cfg = SHAPES[name]
        d = make_synth(name, seed=5)
        nind = cfg["sampling_hops"] + 1
        args = type("A", (), dict(sampling_hops=cfg["sampling_hops"], num_samples=cfg["num_samples"],
                                  use_indicators=True))()
        torch.manual_seed(5)
        gcn_gf = GCN(d.num_features + nind, [256, 1]).to(dev)
        g = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=dev)
        narrow = GCN(d.num_features, [d.num_classes - 1, d.num_classes]).to(dev).eval()       # D <= C
        one = E.evaluate(narrow, gcn_gf, d, args, g, None, nind, dev, mask=d.test_mask, full_batch=True)
        dp = E.evaluate(narrow, gcn_gf, d, args, g, None, nind, dev, mask=d.test_mask, full_batch=True, group=G)
        built = getattr(g, "_sharded_eval", None) is not None
        gcn_c = GCN(d.num_features, [256, d.num_classes]).to(dev).eval()
        idx = d.test_mask.nonzero().squeeze(1)
        loader = [(b,) for b in torch.split(idx, cfg["batch_size"])]      # an odd tail batch on every shape
        one_mb = E.evaluate(gcn_c, gcn_gf, d, args, g, None, nind, dev, mask=d.test_mask, loader=loader,
                            full_batch=False, return_predictions=True)
        dp_mb = E.evaluate(gcn_c, gcn_gf, d, args, g, None, nind, dev, mask=d.test_mask, loader=loader,
                           full_batch=False, return_predictions=True, group=G)
        res[name] = dict(one=one, dp=dp, built=built, one_mb=one_mb[:2], dp_mb=dp_mb[:2],
                         same_preds=bool(torch.equal(one_mb[2], dp_mb[2])), batches=len(loader))
    out[rank] = res
    dist.barrier()
    dist.destroy_process_group()


def test_fallback_and_mini_batch_split_on_one_device(cuda_device):
    world = 2
    out = mp.get_context("spawn").Manager().dict()
    mp.spawn(_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    for r in range(world):
        for name, got in out[r].items():
            assert got["dp"] == got["one"] and not got["built"], (r, name, got)
            assert got["dp_mb"] == got["one_mb"] and got["same_preds"], (r, name, got)
