"""torchrun --nproc-per-node 2 scripts/check_dp_embed.py
Data parallelism with learned node features (--embed_nodes, /root/reference/main.py:89-100,116): the table is replicated,
every rank ships its row-sparse table gradient (the step's all_nodes rows) and every rank applies the same dense Adam to
the mean over ranks.  Checked for both exchanges ('peer': payload pushed inside the step tail, 'nccl': all-gather):
  1. first step: the union of the applied rows == union of the ranks' oracle all_nodes, the applied mean rows == mean of
     the ranks' float64 oracle d loss_c / d x (the per-row bar of tests/test_gpu_embed.py);
  2. three steps against an oracle that applies opt_c / opt_gf to the all-gathered mean gradient: the table within
     Adam's sign-flip bound, rows no rank touched bit-identical to the start;
  3. table, both table moments, parameters and step counts bit-identical across ranks after eager and graph-replayed
     steps (device-side noise);
  4. both ranks on the same batches: (g + g) / 2 == g, so everything is bit-identical to a single-GPU engine;
  5. (peer) a failed exchange is flagged and leaves table, moments and step counts untouched;
  6. the peer and NCCL exchanges agree within the sign-flip bound;
and train() with embed_nodes=True returns with the same table on every rank."""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from grapes_b200.dist import shard_batches                       # noqa: E402
from grapes_b200.engine import GrapesEngine                      # noqa: E402
from grapes_b200.graph import DeviceGraph                        # noqa: E402
from grapes_b200.synth import SHAPES, make_synth                 # noqa: E402
from oracle import reference_port as rp                          # noqa: E402  (test infrastructure)
from parity_utils import _grad_ok                                # noqa: E402

LR_GC = 1e-3
PS_FAILED = 3


def gather(t):
    out = [torch.empty_like(t) for _ in range(dist.get_world_size())]
    dist.all_gather(out, t.contiguous())
    return out


def same_everywhere(tag, tensors):
    for name, t in tensors.items():
        for r, o in enumerate(gather(t)):
            assert torch.equal(o, t), f"{tag}: {name} of rank {r} differs from this rank"


def oracle_params(st):
    return list(st.gcn_c.parameters()) + [st.x] + list(st.gcn_gf.parameters()) + list(st.gcn_z.parameters())


def oracle_dp_step(st, t, noise, dev):
    """reference_step's gradients on this rank's batch, then opt_c / opt_gf on the mean over ranks (rank order)."""
    ref = rp.reference_step(st, t, gumbel_noise=noise, apply_optim=False)
    ps = oracle_params(st)
    flat = torch.cat([(p.grad if p.grad is not None else torch.zeros_like(p)).reshape(-1) for p in ps]).to(dev)
    allg = gather(flat)
    mean = allg[0].clone()
    for g in allg[1:]:
        mean += g
    mean = (mean / len(allg)).cpu()
    off = 0
    for p in ps:
        p.grad = mean[off:off + p.numel()].view_as(p).to(p.dtype).clone()
        off += p.numel()
    st.opt_c.step()
    st.opt_gf.step()
    return ref


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = torch.device("cuda", int(os.environ["LOCAL_RANK"]))
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    cfg = SHAPES["small"]
    d = make_synth("small", seed=4)
    N = d.num_nodes
    B, k, H = cfg["batch_size"], cfg["num_samples"], cfg["sampling_hops"]
    tr = d.train_mask.nonzero().squeeze(1)
    mine = shard_batches(tr.numel() // B, rank, world)
    batch = lambda i: tr[i * B:(i + 1) * B]                       # noqa: E731
    g = DeviceGraph.from_edge_index(d.edge_index, N, device=dev)

    def oracle(dtype):
        return rp.OracleState(d, sampling_hops=H, num_samples=k, seed=107, dtype=dtype, embed_nodes=True)

    def engine(exchange, x=None):
        st = oracle(torch.float64)
        e = GrapesEngine(g, (d.x if x is None else x).to(dev).clone(), d.y.to(dev), num_classes=d.num_classes,
                         batch_size=B, num_samples=k, sampling_hops=H, seed=5, use_tensor_cores=False, embed_nodes=True,
                         lr_gc=LR_GC)
        e.load_state_dicts(gcn_c=st.gcn_c.state_dict(), gcn_gf=st.gcn_gf.state_dict(), gcn_z=st.gcn_z.state_dict())
        if exchange is not None:
            e.enable_data_parallel(exchange=exchange)
        return st, e

    def state_of(e):
        return {"table": e.x, "table_exp_avg": e.emb_exp_avg, "table_exp_avg_sq": e.emb_exp_avg_sq, "params": e.params,
                "exp_avg": e.exp_avg, "exp_avg_sq": e.exp_avg_sq, "steps": e.adam_steps}

    finals, keep = {}, None
    for exchange in ("peer", "nccl"):
        st, eng = engine(exchange)
        st32 = oracle(torch.float32)
        if exchange == "peer":
            assert eng.peer is not None, "peer exchange fell back to NCCL on this box"
        x0 = eng.x.clone()
        touched = torch.zeros(N, dtype=torch.bool, device=dev)
        # ---- 1 + 2: three eager steps with injected noise against the data-parallel oracle ----
        torch.manual_seed(2000 + rank)
        for i in range(3):
            t = batch(mine[i])
            ref = oracle_dp_step(st, t, None, dev)
            noise = [h["noise"] for h in ref["hops"]]
            st32_ref = oracle_dp_step(st32, t, noise, dev)
            rec = eng.step(t.to(dev), gumbel_noise=[None if n is None else n.float().to(dev) for n in noise],
                           apply_optim=True, record=True)
            eng.check_overflow()
            union = rec["embed_union"].long()
            touched[union] = True
            if i > 0:
                continue
            for a, b in zip(rec["hops"], ref["hops"]):
                assert torch.equal(a["sampled"].cpu().long(), b["sampled"]), f"{exchange}: sampled set differs from the oracle"
            an = torch.zeros(N, dtype=torch.int32, device=dev)
            an[ref["all_nodes"].to(dev)] = 1
            an_all = torch.stack(gather(an)).amax(0)
            want_union = an_all.nonzero().squeeze(1)
            assert torch.equal(union, want_union), f"{exchange}: union of the applied rows != union of oracle all_nodes"
            gx = torch.stack(gather(ref["grad_x"].to(dev))).mean(0)
            gx32 = torch.stack(gather(st32_ref["grad_x"].to(dev).double())).mean(0)
            assert _grad_ok(rec["embed_mean_rows"], gx[union].cpu(), gx32[union].cpu(), ()), \
                f"{exchange}: applied mean rows vs mean of the oracle table gradients"
        nsteps = 3
        got, want = eng.x.double().cpu(), st.x.detach().double()
        err = (got - want).abs()
        assert err.max() <= 2.0 * LR_GC * nsteps * 1.01, f"{exchange}: table beyond the Adam sign-flip bound ({err.max():.3e})"
        tch = touched.cpu()
        scale = want.abs().max()
        frac = (err[tch] > 1e-4 * scale).double().mean().item()
        frac32 = ((st32.x.detach().double() - want).abs()[tch] > 1e-4 * scale).double().mean().item()
        assert frac <= max(0.01, 3.0 * frac32), f"{exchange}: {frac:.4f} of the touched table entries off by > 1e-4"
        assert torch.equal(eng.x[~touched], x0[~touched]), f"{exchange}: a row no rank touched moved"
        assert float(eng.adam_steps[0]) == nsteps
        same_everywhere(f"{exchange} eager", state_of(eng))
        # ---- 3: graph-replayed steps, device-side noise ----
        for i in range(3, 9):
            eng.step(batch(mine[i % len(mine)]).to(dev).to(torch.int32).contiguous(), use_graph=True)
        torch.cuda.synchronize()
        eng.check_overflow()
        eng.raise_on_flags(eng.scalars()["flags"])
        assert float(eng.adam_steps[0]) == 9.0 and float(eng.adam_steps[1]) == 9.0
        same_everywhere(f"{exchange} graph replay", state_of(eng))
        finals[exchange] = eng.x.clone()

        # ---- 4: the same batches on every rank == one GPU ----
        _, dp = engine(exchange)
        _, one = engine(None, x=dp.x.cpu())
        same = [tr[i * B:(i + 1) * B].to(dev).to(torch.int32).contiguous() for i in range(5)]
        for i, t in enumerate(same):
            for e in (dp, one):
                e.step(t, use_graph=i >= 2)
        torch.cuda.synchronize()
        dp.check_overflow()
        one.check_overflow()
        for name, t in state_of(dp).items():
            assert torch.equal(t, state_of(one)[name]), f"{exchange}: same batches on every rank: {name} != one GPU"
        assert not torch.equal(dp.x, x0)
        del dp, one
        if exchange == "peer":
            keep = eng

    # ---- 6: peer vs NCCL ----
    diff = (finals["peer"] - finals["nccl"]).abs()
    assert diff.max().item() <= 2.0 * LR_GC * 9 * 1.01, f"peer vs nccl table: {diff.max().item():.3e} beyond the sign-flip bound"

    # ---- 5: a failed exchange (sticky failure word set on every rank: nobody waits) ----
    eng = keep
    dist.barrier()
    eng.peer.state[PS_FAILED] = 1
    torch.cuda.synchronize()
    before = {n: t.clone() for n, t in state_of(eng).items()}
    eng.step(batch(mine[0]).to(dev), apply_optim=True)
    torch.cuda.synchronize()
    assert int(eng.scalars()["flags"]) & 32, "failed exchange not reported in the step's flag word"
    for n, t in state_of(eng).items():
        assert torch.equal(before[n], t), f"a failed exchange changed {n}"
    dist.barrier()

    # ---- train() end to end ----
    from grapes_b200.args import Arguments
    from grapes_b200.train import train
    a = Arguments()
    a.dataset, a.max_epochs, a.batch_size, a.num_samples, a.sampling_hops = "tiny", 1, 32, 8, 2
    a.eval_frequency, a.node_emb_dim, a.embed_nodes = 1, 16, True
    dt = make_synth("tiny", seed=0, features=False)
    dt.num_features = 0
    f1, *_ = train(a, data=dt, device=dev)
    te = train.last_engine
    assert te.dp_world == world and 0.0 <= f1 <= 1.0
    assert float(te.adam_steps[0]) == len(shard_batches((120 + 31) // 32, rank, world))
    same_everywhere("train()", {"table": te.x, "params": te.params})
    dist.barrier()
    if rank == 0:
        print(f"dp embed ok: world={world}; peer vs nccl table max diff {diff.max().item():.3e}", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    try:
        main()
    except BaseException:
        import traceback
        print("RANK", os.environ.get("RANK"), "FAILED:\n" + traceback.format_exc(), flush=True)
        raise
