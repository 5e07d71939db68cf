"""torchrun --nproc-per-node 2 scripts/check_dp_checkpoint.py
Checkpoint and resume of data-parallel train() with learned node features, for both exchanges ("peer", "nccl"), with the
table replicated and sharded across the ranks (shard_embeddings):
  1. train() for two epochs straight through equals train() for one epoch with a checkpoint followed by a resumed
     train() to two epochs: test_f1, every step's log, parameters, the table and its moments, on both ranks;
  2. the W = 2 sharded checkpoint, loaded by one process into a replicated engine, evaluates (full batch) to the scores
     of the W = 2 evaluation.
Prints "dp checkpoint ok" on rank 0."""
import os
import shutil
import sys
import tempfile
import warnings

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from grapes_b200 import checkpoint as C                          # noqa: E402
from grapes_b200 import train as T                               # noqa: E402
from grapes_b200.args import Arguments                           # noqa: E402
from grapes_b200.engine import GrapesEngine                      # noqa: E402
from grapes_b200.graph import DeviceGraph                        # noqa: E402
from grapes_b200.synth import make_synth                         # noqa: E402


def _args(epochs):
    a = Arguments()
    a.dataset, a.max_epochs, a.batch_size, a.num_samples, a.sampling_hops = "small", epochs, 128, 32, 3
    a.embed_nodes, a.node_emb_dim, a.eval_frequency, a.eval_full_batch, a.seed = True, 64, 1, True, 3
    return a


def _run(root, epochs, exchange, shard, resume=False):
    logs = []
    f1, *_ = T.train(_args(epochs), data=make_synth("small", seed=2), device=torch.device("cuda", dist.get_rank()),
                     exchange=exchange, shard_embeddings=shard, step_log=logs.append, checkpoint_dir=root,
                     resume=resume)
    eng = T.train.last_engine
    if eng.embed_shards is not None:
        table, (m, v) = eng.embed_shards.to_dense(), eng.embed_shards.moments_dense()
    else:
        table, m, v = eng.x.clone(), eng.emb_exp_avg.clone(), eng.emb_exp_avg_sq.clone()
    return dict(f1=f1, logs=logs, params=eng.params.clone(), table=table, m=m, v=v)


def _same(a, b, where):
    assert a["f1"] == b["f1"], (where, a["f1"], b["f1"])
    assert a["logs"] == b["logs"], where
    for k in ("params", "table", "m", "v"):
        assert torch.equal(a[k].view(torch.int32), b[k].view(torch.int32)), f"{where}: {k} differs"


def _one_process_eval(path, want_f1):
    """Rank 0 alone: the W = 2 sharded checkpoint in a replicated engine, full-batch evaluation of the test split."""
    dev = torch.device("cuda", 0)
    d = make_synth("small", seed=2)
    a = _args(2)
    meta = C.read_meta(path)
    g = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=dev)
    x = torch.zeros(meta["N"], meta["F"], device=dev)
    eng = GrapesEngine(g, x, d.y.to(dev), num_classes=d.num_classes, batch_size=a.batch_size,
                       num_samples=a.num_samples, sampling_hops=a.sampling_hops, hidden_dim=a.hidden_dim, seed=99,
                       embed_nodes=True)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")                 # world 2 -> 1, shard_embeddings True -> False
        C.load(eng, path, args=a, group=None)
    d.x = eng.x
    _, f1 = T.evaluate(eng, d, d.test_mask.to(dev), full_batch=True, args=a)
    assert f1 == want_f1, (f1, want_f1)


def main():
    rank = int(os.environ.get("RANK", "0"))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", rank))
    box = [tempfile.mkdtemp(prefix="grapes_dp_ckpt_") if rank == 0 else None]
    dist.broadcast_object_list(box, src=0)
    base = box[0]
    try:
        for exchange in ("peer", "nccl"):
            for shard in (False, True):
                tag = f"{exchange} {'sharded' if shard else 'replicated'}"
                want = _run(os.path.join(base, f"{exchange}{shard}_straight"), 2, exchange, shard)
                root = os.path.join(base, f"{exchange}{shard}")
                first = _run(root, 1, exchange, shard)
                got = _run(root, 2, exchange, shard, resume=True)
                got["logs"] = first["logs"] + got["logs"]
                _same(got, want, tag)
                print(f"rank {rank} {tag}: interrupted and resumed train() == straight, test_f1 {want['f1']}", flush=True)
                if shard and exchange == "peer":
                    dist.barrier()
                    if rank == 0:
                        _one_process_eval(C.latest(root), want["f1"])
                        print("rank 0: W = 2 sharded checkpoint evaluated by one process: same scores", flush=True)
                    dist.barrier()
    finally:
        dist.barrier()
        if rank == 0:
            shutil.rmtree(base, ignore_errors=True)
    if rank == 0:
        print("dp checkpoint ok", flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
