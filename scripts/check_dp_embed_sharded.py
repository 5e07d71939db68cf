"""torchrun --nproc-per-node 2 scripts/check_dp_embed_sharded.py
A learned node-feature table sharded by rows with its Adam moments (``dist.ShardedEmbedding``, ``train(...,
shard_embeddings=True)``) against the replicated learned table, for both exchanges ("peer" and "nccl"):
  1. train() with and without shard_embeddings: bit-identical parameters, gathered table and moments, the same test_f1;
     each rank holds about 3 * ceil(N / W) * F * 4 bytes of table and moments;
  2. ordering: eager engine steps with rank 1's table merge delayed (torch.cuda._sleep ahead of it on the engine's stream)
     stay bit-identical to the replicated engine;
  3. sensitivity: the same delayed run with the epoch wait patched out differs (the check can see the hazard);
  4. missing post (peer exchange): rank 1 skips one epoch post; rank 0's bounded wait flags GRAPES_OVF_PEER_TIMEOUT, its
     step is not applied and the step's flag check raises.
Prints "dp embed sharded ok" on rank 0."""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from grapes_b200._lib import GrapesError                         # noqa: E402
from grapes_b200.dist import ShardedEmbedding, shard_batches     # noqa: E402
from grapes_b200.engine import GrapesEngine                      # noqa: E402
from grapes_b200.graph import DeviceGraph                        # noqa: E402
from grapes_b200.synth import SHAPES, make_synth                 # noqa: E402

DELAY_CYCLES = 200_000_000                                       # ~0.1 s on a B200


def _train_runs(rank, world, dev, exchange):
    from grapes_b200 import train as T
    from grapes_b200.args import Arguments
    out = []
    for shard in (True, False):
        a = Arguments()
        a.dataset, a.max_epochs, a.batch_size, a.num_samples, a.sampling_hops = "small", 2, 128, 32, 3
        a.embed_nodes, a.node_emb_dim, a.eval_frequency, a.eval_full_batch = True, 64, 1, True
        f1, *_ = T.train(a, data=make_synth("small", seed=2), device=dev, exchange=exchange, shard_embeddings=shard)
        eng = T.train.last_engine
        assert (eng.embed_shards is not None) == shard
        if shard:
            es = eng.embed_shards
            table, (m, v) = es.to_dense(), es.moments_dense()
            held = es.table_bytes + es.moment_bytes
            want = 3 * -(-es.N // world) * es.F * 4
            assert want <= held <= want + 3 * es.F * 4, (held, want)
            print(f"rank {rank} {exchange}: table + moments {held} bytes on this rank "
                  f"(replicated {3 * es.N * es.F * 4})", flush=True)
        else:
            table, m, v = eng.x.clone(), eng.emb_exp_avg.clone(), eng.emb_exp_avg_sq.clone()
        out.append((f1, eng.params.clone(), table, m, v))
    (f1s, ps, ts, ms, vs), (f1r, pr, tr, mr, vr) = out
    assert f1s == f1r, (exchange, f1s, f1r)
    for name, a, b in (("params", ps, pr), ("table", ts, tr), ("exp_avg", ms, mr), ("exp_avg_sq", vs, vr)):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32)), f"{exchange}: {name} differs"
    print(f"rank {rank} {exchange}: train() sharded == replicated, test_f1 {f1s}", flush=True)


def _engine(d, g, x, dev, sharded, exchange):
    cfg = SHAPES["small"]
    xin = ShardedEmbedding(x, dev) if sharded else x.to(dev)
    eng = GrapesEngine(g, xin, d.y.to(dev), num_classes=d.num_classes, batch_size=cfg["batch_size"],
                       num_samples=cfg["num_samples"], sampling_hops=cfg["sampling_hops"], hidden_dim=256, seed=5,
                       embed_nodes=True)
    eng.enable_data_parallel(exchange=exchange)
    return eng


def _state(eng):
    if eng.embed_shards is None:
        return eng.params.clone(), eng.x.clone()
    return eng.params.clone(), eng.embed_shards.to_dense()


def _ordering(rank, world, dev, exchange):
    d = make_synth("small", seed=3)
    g = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=dev)
    x = torch.empty(d.num_nodes, 64).normal_(generator=torch.Generator().manual_seed(4))
    idx = d.train_mask.nonzero().squeeze(1).to(torch.int32).to(dev)
    batches = [b.contiguous() for b in torch.split(idx, SHAPES["small"]["batch_size"])]
    batches = [batches[i] for i in shard_batches(len(batches), rank, world)][:5]
    real_merge, real_wait = GrapesEngine._enqueue_embed_merge, GrapesEngine._enqueue_epoch_wait

    def delayed_merge(self, *a):
        if rank == 1:
            torch.cuda._sleep(DELAY_CYCLES)
        real_merge(self, *a)

    def run(sharded, delay=False, wait=True):
        eng = _engine(d, g, x, dev, sharded, exchange)
        GrapesEngine._enqueue_embed_merge = delayed_merge if delay else real_merge
        GrapesEngine._enqueue_epoch_wait = real_wait if wait else (lambda self, ctx, st: None)
        try:
            for b in batches:
                eng.step(b)
            torch.cuda.synchronize()
            eng.check_overflow()
        finally:
            GrapesEngine._enqueue_embed_merge, GrapesEngine._enqueue_epoch_wait = real_merge, real_wait
        out = _state(eng)
        dist.barrier()
        return out

    rep = run(False)
    ordered = run(True, delay=True)
    for a, b in zip(rep, ordered):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32)), f"{exchange}: delayed merge changed the result"
    unordered = run(True, delay=True, wait=False)
    same = all(torch.equal(a.view(torch.int32), b.view(torch.int32)) for a, b in zip(rep, unordered))
    flag = torch.tensor([0 if same else 1], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MAX)
    assert int(flag.item()) == 1, f"{exchange}: without the epoch wait the delayed run still matched: the check is blind"
    print(f"rank {rank} {exchange}: delayed merge bit-identical with the wait, differs without it", flush=True)
    return d, g, x, batches


def _missing_post(rank, dev, d, g, x, batches):
    eng = _engine(d, g, x, dev, True, "peer")
    eng.epoch_spin_limit = 20000
    eng.step(batches[0])
    torch.cuda.synchronize()
    eng.check_overflow()
    dist.barrier()
    if rank == 1:
        real = eng.L.grapes_embed_epoch_post
        calls = []

        def skip_once(*a):
            if not calls:
                calls.append(1)
                return
            real(*a)
        eng.L.grapes_embed_epoch_post = skip_once
    try:
        eng.step(batches[1])                          # rank 1 does not post this step's epoch
        torch.cuda.synchronize()
        dist.barrier()
        before = eng.params.clone()
        eng.step(batches[2])                          # rank 0 waits for it: bounded, flagged, not applied
        torch.cuda.synchronize()
    finally:
        if rank == 1:
            del eng.L.grapes_embed_epoch_post
    if rank == 0:
        assert int(eng.overflow.item()) & 32, "the missing post was not flagged"
        assert torch.equal(before, eng.params), "the step was applied after a missing post"
        try:
            eng.raise_on_flags(int(eng.scalars()["flags"]))
            raise AssertionError("the step's flags did not raise")
        except GrapesError as exc:
            assert "exchange failed" in str(exc), str(exc)
        print("rank 0: missing post flagged, step not applied, flags raise", flush=True)
    dist.barrier()


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = torch.device("cuda", int(os.environ["LOCAL_RANK"]))
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    for exchange in ("peer", "nccl"):
        _train_runs(rank, world, dev, exchange)
        d, g, x, batches = _ordering(rank, world, dev, exchange)
    _missing_post(rank, dev, d, g, x, batches)
    dist.barrier()
    if rank == 0:
        print(f"dp embed sharded ok: world={world}", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    try:
        main()
    except BaseException:
        import traceback
        print("RANK", os.environ.get("RANK"), "FAILED:\n" + traceback.format_exc(), flush=True)
        raise
