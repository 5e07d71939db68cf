"""torchrun --nproc-per-node 2 scripts/check_dp_full_batch.py
Data-parallel full-graph training (``full_batch.train(..., group=...)``) over a real group, against itself and the
one-process emulation:
  1. the parameters are bit-identical across the ranks after every epoch;
  2. the trained parameters are bit-identical to ``train_emulated`` with the same number of ranks, in one process;
  3. the test F1 equals a single-process ``evaluate()`` of the final model;
  4. the window structure is built once per run (the evaluations reuse the training's), and dropped on return;
  5. a peer row table that cannot be mapped on one rank is refused on both.
Cases: a directed graph with reg_param (F <= D) and a cora-shaped graph (F > D, the d pre table).
Prints "dp full batch ok" on rank 0."""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import grapes_b200.dist as D                                     # noqa: E402
from grapes_b200 import full_batch as fb                         # noqa: E402
from grapes_b200 import gcn as G                                 # noqa: E402
from grapes_b200._lib import GrapesError                         # noqa: E402
from grapes_b200.args import Arguments                           # noqa: E402
from grapes_b200.eval import evaluate                            # noqa: E402
from grapes_b200.graph import DeviceGraph                        # noqa: E402
from grapes_b200.synth import make_synth                         # noqa: E402
from directed_utils import directed_synth                        # noqa: E402


def gather_equal(t, group):
    parts = [torch.empty_like(t) for _ in range(dist.get_world_size(group))]
    dist.all_gather(parts, t.contiguous(), group=group)
    return all(torch.equal(p, parts[0]) for p in parts)


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = torch.device("cuda", int(os.environ["LOCAL_RANK"]))
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    grp = dist.group.WORLD
    builds = []
    real_build = G.ShardedGraphNorm.__init__

    def counting(self, *a, **kw):
        builds.append(1)
        real_build(self, *a, **kw)
    G.ShardedGraphNorm.__init__ = counting
    real_step = torch.optim.Adam.step
    per_epoch = []

    def checked_step(self, *a, **kw):
        out = real_step(self, *a, **kw)
        if getattr(self, "_dp_check", True):
            flat = torch.cat([p.detach().reshape(-1) for grp_ in self.param_groups for p in grp_["params"]])
            per_epoch.append(gather_equal(flat, grp))
        return out
    torch.optim.Adam.step = checked_step
    try:
        for name in ("directed", "cora"):
            d = directed_synth("small", 3) if name == "directed" else make_synth("cora", seed=5)
            args = Arguments(dataset="synth", hidden_dim=32 if name == "directed" else 16, max_epochs=4,
                             eval_frequency=2, seed=4, lr_gc=1e-2, reg_param=1e-3 if name == "directed" else 0.)
            builds.clear(), per_epoch.clear()
            f1, *_ = fb.train(args, data=d, device=dev, group=grp)
            model = fb.train.last_model
            assert len(per_epoch) == args.max_epochs and all(per_epoch), f"{name}: parameters differ across ranks"
            assert len(builds) == 1, f"{name}: window structure built {len(builds)} times"
            params = {n: p.detach().clone() for n, p in model.named_parameters()}
            torch.optim.Adam.step = real_step
            G.ShardedGraphNorm.__init__ = real_build
            fb.train_emulated(args, d, dev, world)
            torch.optim.Adam.step = checked_step
            G.ShardedGraphNorm.__init__ = counting
            for n, p in fb.train.last_model.named_parameters():
                assert torch.equal(params[n], p.detach()), f"{name}: {n} differs from the emulated run"
            g = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=dev)
            _, one = evaluate(model, None, d, args, g, None, 0, dev, mask=d.test_mask, eval_on_cpu=False,
                              full_batch=True)
            assert one == f1, (name, one, f1)
            print(f"rank {rank} {name}: test_f1 {f1}", flush=True)
    finally:
        torch.optim.Adam.step = real_step
        G.ShardedGraphNorm.__init__ = real_build

    # a peer row table that cannot be mapped on rank 1: refused on both ranks
    real_table = D.PeerRowTable.__init__

    def failing(self, *a, **kw):
        if dist.get_rank() == 1:
            raise RuntimeError("forced mapping failure")
        real_table(self, *a, **kw)
    D.PeerRowTable.__init__ = failing
    try:
        fb.train(Arguments(dataset="synth", hidden_dim=32, max_epochs=1), data=make_synth("small", seed=1), device=dev,
                 group=grp)
        raise AssertionError("an unmappable row table was not refused")
    except GrapesError as exc:
        assert "row table" in str(exc), exc
    finally:
        D.PeerRowTable.__init__ = real_table
    dist.barrier()
    if rank == 0:
        print(f"dp full batch ok: world={world}", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    try:
        main()
    except BaseException:
        import traceback
        print("RANK", os.environ.get("RANK"), "FAILED:\n" + traceback.format_exc(), flush=True)
        raise
