"""torchrun --nproc-per-node 2 scripts/check_dp_dropout.py
Data parallelism with dropout in the classifier GCN (--dropout 0.5, modules/gcn.py:33,37): every rank draws its own masks
(the rank is part of the Philox counter), and the exchanged gradient is the mean of the ranks' gradients, each taken
through that rank's masks.  For both exchanges ('peer', 'nccl'), with and without learned node features:
  1. each rank's recorded masks equal the numpy restatement for its rank, and the ranks' masks differ;
  2. the exchanged (mean) gradient of all three networks -- and of the table rows with --embed_nodes -- equals the mean
     of the ranks' float64 oracle gradients, each computed with that rank's masks replayed (1e-5 bar of
     tests/parity_utils.py);
  3. parameters, moments, mask counters (and the table) are bit-identical across ranks after the eager step and after
     graph-replayed steps."""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from dropout_utils import engine_masks, keep_mask, replay_masks, tag, threshold   # noqa: E402
from grapes_b200.dist import shard_batches                       # noqa: E402
from grapes_b200.engine import GrapesEngine                      # noqa: E402
from grapes_b200.graph import DeviceGraph                        # noqa: E402
from grapes_b200.synth import SHAPES, make_synth                 # noqa: E402
from oracle import reference_port as rp                          # noqa: E402  (test infrastructure)
from parity_utils import _grad_ok                                # noqa: E402

P, SEED = 0.5, 5


def gather(t):
    out = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(out, t.contiguous())
    return out


def mean_over_ranks(t, dev):
    """rank-order mean of a host tensor, back on the host as float64"""
    return torch.stack(gather(t.to(dev).double())).mean(0).cpu()


def same_everywhere(what, tensors):
    for name, t in tensors.items():
        for r, o in enumerate(gather(t)):
            assert torch.equal(o, t), f"{what}: {name} of rank {r} differs from this rank"


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = torch.device("cuda", int(os.environ["LOCAL_RANK"]))
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    cfg = SHAPES["small"]
    d = make_synth("small", seed=4)
    B, k, H = cfg["batch_size"], cfg["num_samples"], cfg["sampling_hops"]
    tr = d.train_mask.nonzero().squeeze(1)
    mine = shard_batches(tr.numel() // B, rank, world)
    batch = lambda i: tr[i * B:(i + 1) * B]                       # noqa: E731
    g = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=dev)
    thr = threshold(P)

    for exchange in ("peer", "nccl"):
        for embed in (False, True):
            what = f"{exchange}{' embed_nodes' if embed else ''}"
            kw = dict(sampling_hops=H, num_samples=k, seed=107, embed_nodes=embed, dropout=P)
            st, st32 = rp.OracleState(d, dtype=torch.float64, **kw), rp.OracleState(d, dtype=torch.float32, **kw)
            eng = GrapesEngine(g, d.x.to(dev).clone(), d.y.to(dev), num_classes=d.num_classes, batch_size=B,
                               num_samples=k, sampling_hops=H, seed=SEED, use_tensor_cores=False, embed_nodes=embed,
                               dropout=P)
            eng.load_state_dicts(gcn_c=st.gcn_c.state_dict(), gcn_gf=st.gcn_gf.state_dict(), gcn_z=st.gcn_z.state_dict())
            eng.enable_data_parallel(exchange=exchange)
            if exchange == "peer":
                assert eng.peer is not None, "peer exchange fell back to NCCL on this box"
            # ---- first step: this rank's masks replayed in the oracle ----
            torch.manual_seed(3000 + rank)
            t = batch(mine[0])
            with replay_masks(engine_masks(SEED, 0, P, rank)):
                ref = rp.reference_step(st, t, apply_optim=False)
                noise = [h["noise"] for h in ref["hops"]]
                ref32 = rp.reference_step(st32, t, gumbel_noise=noise, apply_optim=False)
            rec = eng.step(t.to(dev), gumbel_noise=[None if n is None else n.float().to(dev) for n in noise],
                           apply_optim=True, record=True)
            eng.check_overflow()
            A = rec["all_nodes"].numel()
            assert torch.equal(rec["all_nodes"].cpu().long(), ref["all_nodes"]), f"{what}: all_nodes"
            for site, width in ((0, eng.D), (1, eng.C)):
                got = rec["dropout_keep"][site].cpu().numpy()
                assert (got == keep_mask(SEED, 0, tag(site, rank), thr, A, width)).all(), f"{what}: site {site} mask"
            head = rec["dropout_keep"][0][:16].to(torch.uint8)
            heads = gather(head)
            assert all(not torch.equal(heads[0], h) for h in heads[1:]), f"{what}: ranks drew the same hidden mask"
            # ---- the exchanged gradient = mean of the ranks' oracle gradients ----
            for net, key in (("gcn_c", "grads_c"), ("gcn_gf", "grads_gf"), ("gcn_z", "grads_z")):
                for name, gref in ref[key].items():
                    if gref is None:
                        continue
                    want, want32 = mean_over_ranks(gref, dev), mean_over_ranks(ref32[key][name], dev)
                    assert _grad_ok(rec["grads"][net][name], want, want32, ()), f"{what}: mean gradient {net}.{name}"
            if embed:
                union = rec["embed_union"].long().cpu()
                gx, gx32 = mean_over_ranks(ref["grad_x"], dev), mean_over_ranks(ref32["grad_x"], dev)
                assert _grad_ok(rec["embed_mean_rows"], gx[union], gx32[union], ()), f"{what}: mean table rows"
            state = {"params": eng.params, "exp_avg": eng.exp_avg, "exp_avg_sq": eng.exp_avg_sq,
                     "steps": eng.adam_steps, "drop_state": eng.drop_state}
            if embed:
                state.update(table=eng.x, table_exp_avg=eng.emb_exp_avg, table_exp_avg_sq=eng.emb_exp_avg_sq)
            same_everywhere(f"{what} eager", state)
            # ---- graph-replayed steps, device-side noise ----
            for i in range(1, 7):
                eng.step(batch(mine[i % len(mine)]).to(dev).to(torch.int32).contiguous(), use_graph=True)
            torch.cuda.synchronize()
            eng.check_overflow()
            eng.raise_on_flags(eng.scalars()["flags"])
            assert int(eng.drop_state[1]) == 7 and float(eng.adam_steps[0]) == 7.0
            same_everywhere(f"{what} graph replay", state)
            del eng
            dist.barrier()
    if rank == 0:
        print(f"dp dropout ok: world={world}", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    try:
        main()
    except BaseException:
        import traceback
        print("RANK", os.environ.get("RANK"), "FAILED:\n" + traceback.format_exc(), flush=True)
        raise
