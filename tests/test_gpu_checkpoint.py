"""Checkpoint and resume on one B200 (``grapes_b200.checkpoint``, ``train(..., checkpoint_dir=, resume=)``):

* 2K steps straight through equal K steps, save, a fresh engine built with a different seed (and table), load, K more
  steps: parameters, both Adam states, both Philox counters, the learned table and its moments and every step's
  ``scal_stats`` read-back bit for bit -- for trajectory balance, REINFORCE, random sampling, multi-label, dropout,
  learned node features, a bf16 table, the SIMT engine and graph replay with cross-step prefetch;
* a graph captured before the load replays the loaded state (nothing is rebound);
* the resume leg in a separate process;
* an emulated sharded learned table (W = 2, 3, 8) loaded into a replicated engine and into an emulated W' = 3 engine;
* the refusals of save (a flag word, ranks whose parameters differ);
* ``train()`` interrupted (at an epoch end, and mid-epoch with ``checkpoint_every``) and resumed in a new process equals
  the uninterrupted run: test_f1, step log, validation lines, final parameters;
* ``model.pt`` loaded into ``grapes_b200.gcn.GCN`` evaluates to the live engine's scores."""
import logging
import os
import pickle
import socket
import subprocess
import sys
import warnings

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
K = 3
CASES = {"tb": {}, "reinforce": dict(reinforce_baseline=True), "random": dict(random_sampling=True),
         "multilabel": {}, "dropout": dict(dropout=0.5), "embed": dict(embed_nodes=True), "bf16": {},
         "simt": dict(use_tensor_cores=False), "graph": {}}


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t.view(torch.int16) if t.dtype == torch.bfloat16 else t


def _same(a, b, where=""):
    if isinstance(a, dict):
        assert a.keys() == b.keys(), where
        for k in a:
            _same(a[k], b[k], f"{where}.{k}")
    elif isinstance(a, (list, tuple)):
        assert len(a) == len(b), where
        for i, (u, v) in enumerate(zip(a, b)):
            _same(u, v, f"{where}[{i}]")
    elif isinstance(a, torch.Tensor):
        assert a.shape == b.shape and a.dtype == b.dtype, where
        assert torch.equal(_bits(a.cpu().contiguous()), _bits(b.cpu().contiguous())), where
    else:
        assert a == b or (a != a and b != b), f"{where}: {a} != {b}"


def _setup(case, dev, seed, table_seed=4, W=None):
    """The case's engine over the small synthetic graph; ``seed`` (weights and Philox counters) and ``table_seed`` (a
    learned table) differ between the run that saves and the engine that loads.  ``W``: an emulated sharded table."""
    from grapes_b200.dist import ShardedEmbedding
    from grapes_b200.engine import GrapesEngine
    from grapes_b200.graph import DeviceGraph
    from grapes_b200.synth import SHAPES, make_synth
    cfg = SHAPES["small"]
    d = make_synth("small", seed=3, multilabel=case == "multilabel")
    kw = dict(CASES.get(case, {}))
    x = d.x
    if kw.get("embed_nodes") or W is not None:
        kw["embed_nodes"] = True
        x = torch.empty(d.num_nodes, 64).normal_(generator=torch.Generator().manual_seed(table_seed))
    x = x.to(dev)
    if case == "bf16":
        x = x.to(torch.bfloat16)
    if W is not None:
        x = ShardedEmbedding.emulate(x, W)[W - 1]
    g = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=dev)
    eng = GrapesEngine(g, x, d.y.to(dev), num_classes=d.num_classes, batch_size=cfg["batch_size"],
                       num_samples=cfg["num_samples"], sampling_hops=cfg["sampling_hops"], hidden_dim=256, seed=seed,
                       **kw)
    idx = d.train_mask.nonzero().squeeze(1).to(torch.int32).to(dev)
    batches = [b.contiguous() for b in torch.split(idx, cfg["batch_size"])][:2 * K]
    return d, eng, batches


def _run(eng, batches, graph=False, prefetch=False):
    logs = []
    for i, b in enumerate(batches):
        nxt = batches[i + 1] if prefetch and i + 1 < len(batches) else None
        eng.step(b, use_graph=graph, next_targets=nxt)
        logs.append(eng.scal_stats.clone())
    torch.cuda.synchronize()
    eng.check_overflow()
    return logs


def _state(eng):
    out = {n: getattr(eng, n).clone() for n in ("params", "exp_avg", "exp_avg_sq", "adam_steps", "rng_state",
                                                "drop_state")}
    if eng.embed_nodes:
        es = eng.embed_shards
        if es is not None:
            out["table"], (out["table_m"], out["table_v"]) = es.to_dense(), es.moments_dense()
        else:
            out["table"], out["table_m"], out["table_v"] = eng.x.clone(), eng.emb_exp_avg.clone(), eng.emb_exp_avg_sq.clone()
    return out


def _mode(case):
    return dict(graph=True, prefetch=True) if case == "graph" else {}


@pytest.mark.parametrize("case", list(CASES))
def test_resume_is_bit_identical(cuda_device, tmp_path, case):
    from grapes_b200 import checkpoint as C
    dev = cuda_device
    _, a, batches = _setup(case, dev, seed=5)
    want_logs = _run(a, batches, **_mode(case))
    _, b, _ = _setup(case, dev, seed=5)
    logs1 = _run(b, batches[:K], **_mode(case))
    C.save(b, str(tmp_path), dict(step=K))
    _, c, _ = _setup(case, dev, seed=77, table_seed=78)
    assert not torch.equal(c.params, b.params)
    C.load(c, str(tmp_path))
    logs2 = _run(c, batches[K:], **_mode(case))
    _same(_state(a), _state(c), case)
    _same(want_logs, logs1 + logs2, f"{case} scal_stats")


def test_graph_captured_before_load_replays_loaded_state(cuda_device, tmp_path):
    from grapes_b200 import checkpoint as C
    dev = cuda_device
    _, a, batches = _setup("tb", dev, seed=5)
    want_logs = _run(a, batches, graph=True)
    _, b, _ = _setup("tb", dev, seed=5)
    logs1 = _run(b, batches[:K], graph=True)
    C.save(b, str(tmp_path), dict(step=K))
    _, c, _ = _setup("tb", dev, seed=77)
    _run(c, batches[:1], graph=True)                     # captures the step graph with c's own state
    graphs = dict(c._graphs)
    C.load(c, str(tmp_path))
    logs2 = _run(c, batches[K:], graph=True)
    assert c._graphs == graphs                          # the same captured graph replayed every step
    _same(_state(a), _state(c), "graph before load")
    _same(want_logs, logs1 + logs2, "graph before load scal_stats")


def _resume_leg(case, ckpt, out):
    """The resume leg of test_resume_in_a_new_process, run as its own process."""
    from grapes_b200 import checkpoint as C
    dev = torch.device("cuda:0")
    _, c, batches = _setup(case, dev, seed=77, table_seed=78)
    C.load(c, ckpt)
    logs = _run(c, batches[K:], **_mode(case))
    torch.save({"state": {k: v.cpu() for k, v in _state(c).items()}, "logs": [t.cpu() for t in logs]}, out)


def _child(*argv):
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT, os.path.join(ROOT, "tests")]))
    res = subprocess.run([sys.executable, os.path.abspath(__file__), *argv], capture_output=True, text=True, env=env,
                         timeout=900)
    assert res.returncode == 0, res.stdout[-4000:] + res.stderr[-4000:]
    return res


@pytest.mark.parametrize("case", ["embed", "graph"])
def test_resume_in_a_new_process(cuda_device, tmp_path, case):
    from grapes_b200 import checkpoint as C
    dev = cuda_device
    _, a, batches = _setup(case, dev, seed=5)
    want_logs = _run(a, batches, **_mode(case))
    _, b, _ = _setup(case, dev, seed=5)
    logs1 = _run(b, batches[:K], **_mode(case))
    C.save(b, str(tmp_path / "ck"), dict(step=K))
    out = str(tmp_path / "leg2.pt")
    _child("resume", case, str(tmp_path / "ck"), out)
    got = torch.load(out, weights_only=True)
    _same(_state(a), got["state"], f"{case} new process")
    _same([t.cpu() for t in want_logs], [t.cpu() for t in logs1] + got["logs"], f"{case} new process scal_stats")


@pytest.mark.parametrize("W", [2, 3, 8])
def test_sharded_table_resaved_into_other_layouts(cuda_device, tmp_path, W):
    """An emulated W-rank sharded table saved after K steps, loaded into a replicated engine and into an emulated
    W' = 3 engine: the dense table and moments equal the saved ones, and the next K steps equal those of the W engine."""
    from grapes_b200 import checkpoint as C
    dev = cuda_device
    _, a, batches = _setup("embed", dev, seed=5, W=W)
    _run(a, batches[:K])
    path = C.save(a, str(tmp_path), dict(step=K))
    saved = _state(a)
    t, m, v = C.table_source(path)
    _same((t, m, v), (saved["table"], saved["table_m"], saved["table_v"]), f"W {W} files")
    want_logs = _run(a, batches[K:])
    for other in (None, 3):
        _, c, _ = _setup("embed", dev, seed=77, table_seed=78, W=other)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")              # shard_embeddings differs for the replicated engine
            C.load(c, path)
        _same(_state(c), saved, f"W {W} -> {other} loaded")
        _same(_run(c, batches[K:]), want_logs, f"W {W} -> {other} steps")
        _same(_state(c), _state(a), f"W {W} -> {other} after steps")


def test_save_refuses_flags(cuda_device, tmp_path):
    from grapes_b200 import checkpoint as C
    from grapes_b200._lib import GrapesError
    _, a, batches = _setup("tb", cuda_device, seed=5)
    _run(a, batches[:1])
    a.overflow.fill_(4)
    with pytest.raises(GrapesError, match="flag word"):
        C.save(a, str(tmp_path), dict(step=1))
    assert C.latest(str(tmp_path)) is None


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _holder(rank, world, port, root, out):
    import torch.distributed as dist
    from grapes_b200 import checkpoint as C
    from grapes_b200._lib import GrapesError
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    _, e, batches = _setup("tb", torch.device("cuda:0"), seed=5)
    _run(e, batches[:1])
    res = {}
    res["ok"] = C.save(e, root, dict(step=1), group=dist.group.WORLD)
    if rank == 1:
        e.params[7] += 1.0
    try:
        C.save(e, root, dict(step=2), group=dist.group.WORLD)
        res["refused"] = None
    except GrapesError as exc:
        res["refused"] = str(exc)
    out[rank] = res
    dist.barrier()
    dist.destroy_process_group()


def test_save_refuses_parameters_that_differ_between_holders(cuda_device, tmp_path):
    """Two processes on one GPU holding the same engine (gloo group): equal parameters save, a parameter changed on one
    holder is refused on both."""
    import torch.multiprocessing as mp
    out = mp.get_context("spawn").Manager().dict()
    mp.spawn(_holder, args=(2, _free_port(), str(tmp_path), out), nprocs=2, join=True)
    for r in range(2):
        assert out[r]["ok"].endswith("step-000000001")
        assert out[r]["refused"] is not None and "parameters differ" in out[r]["refused"], out[r]["refused"]


# ------------------------------------------------------------------------------------------------ train()
class _Lines(logging.Handler):
    def __init__(self):
        super().__init__()
        self.lines = []

    def emit(self, record):
        self.lines.append(record.getMessage())


def _train(ckpt, max_epochs, embed, die_at=None, **kw):
    """train() on the small graph with the step log and the log lines recorded; ``die_at``: the step log raises at
    that step, as a process that dies."""
    from grapes_b200 import train as T
    from grapes_b200.args import Arguments
    from grapes_b200.synth import make_synth
    a = Arguments()
    a.dataset, a.max_epochs, a.batch_size, a.num_samples, a.sampling_hops = "small", max_epochs, 128, 32, 3
    a.eval_frequency, a.seed = 1, 11
    a.embed_nodes, a.node_emb_dim = embed, 32
    logs, rec = [], _Lines()
    logger = logging.getLogger("grapes_checkpoint_test")
    logger.handlers, logger.propagate = [rec], False
    logger.setLevel("INFO")

    def step_log(d):
        if die_at is not None and len(logs) == die_at:
            raise KeyboardInterrupt("process died")
        logs.append(d)
    get_logger, T.get_logger = T.get_logger, (lambda: logger)
    try:
        f1 = None
        try:
            f1, *_ = T.train(a, data=make_synth("small", seed=2), device=torch.device("cuda:0"), step_log=step_log,
                             checkpoint_dir=ckpt, **kw)
        except KeyboardInterrupt:
            if die_at is None:
                raise
    finally:
        T.get_logger = get_logger
    eng = T.train.last_engine if f1 is not None else None
    st = {k: v.cpu() for k, v in _state(eng).items()} if eng is not None else None
    return dict(f1=f1, logs=logs, valid=[ln for ln in rec.lines if "valid_" in ln], state=st)


def _train_leg(ckpt, max_epochs, embed, every, out):
    r = _train(ckpt, int(max_epochs), embed == "1", checkpoint_every=int(every), resume=True)
    with open(out, "wb") as f:
        pickle.dump(r, f)


@pytest.mark.parametrize("embed", [False, True])
def test_train_resumed_at_an_epoch_end_in_a_new_process(cuda_device, tmp_path, embed):
    from grapes_b200 import checkpoint as C
    want = _train(str(tmp_path / "straight"), 3, embed)
    first = _train(str(tmp_path / "ck"), 1, embed)
    assert C.read_meta(str(tmp_path / "ck"))["epoch"] == 1
    out = str(tmp_path / "leg2.pkl")
    _child("train", str(tmp_path / "ck"), "3", "1" if embed else "0", "0", out)
    with open(out, "rb") as f:
        got = pickle.load(f)
    assert got["f1"] == want["f1"]
    assert first["logs"] + got["logs"] == want["logs"]
    assert first["valid"] + got["valid"] == want["valid"] and len(want["valid"]) == 3
    _same(got["state"], want["state"], "train epoch resume")


def test_train_resumed_mid_epoch_in_a_new_process(cuda_device, tmp_path):
    from grapes_b200 import checkpoint as C
    want = _train(str(tmp_path / "straight"), 2, False, checkpoint_every=4)
    dead = _train(str(tmp_path / "ck"), 2, False, die_at=10, checkpoint_every=4)
    meta = C.read_meta(str(tmp_path / "ck"))
    assert (meta["epoch"], meta["batch"], meta["step"]) == (1, 8, 8)
    out = str(tmp_path / "leg2.pkl")
    _child("train", str(tmp_path / "ck"), "2", "0", "4", out)
    with open(out, "rb") as f:
        got = pickle.load(f)
    assert got["f1"] == want["f1"]
    assert dead["logs"][:8] + got["logs"] == want["logs"]
    assert got["valid"] == want["valid"]
    _same(got["state"], want["state"], "train mid-epoch resume")


def test_model_pt_loads_into_gcn_and_evaluates_like_the_engine(cuda_device, tmp_path):
    from grapes_b200 import checkpoint as C
    from grapes_b200 import eval as E
    from grapes_b200 import train as T
    from grapes_b200.gcn import GCN
    dev = cuda_device
    d, a, batches = _setup("tb", dev, seed=5)
    _run(a, batches)
    path = C.save(a, str(tmp_path), dict(step=2 * K))
    d.x = d.x.to(dev)
    mask = d.test_mask.to(dev)
    want = T.evaluate(a, d, mask, full_batch=True)
    model = torch.load(os.path.join(path, "model.pt"), weights_only=True)
    gcn_c = GCN(a.F, [a.D, a.C]).to(dev)
    gcn_c.load_state_dict(model["gcn_c"])
    gcn_gf = GCN(a.Fp, [a.D, 1]).to(dev)
    gcn_gf.load_state_dict(model["gcn_gf"])
    gcn_z = GCN(a.F, [a.D, 1])
    gcn_z.load_state_dict(model["gcn_z"])
    ns = type("A", (), dict(sampling_hops=a.H, num_samples=a.k, use_indicators=a.use_ind))()
    got = E.evaluate(gcn_c, gcn_gf, d, ns, a.g, None, a.num_ind, dev, mask=mask, eval_on_cpu=False, full_batch=True)
    assert got == want


if __name__ == "__main__":
    if sys.argv[1] == "resume":
        _resume_leg(*sys.argv[2:])
    elif sys.argv[1] == "train":
        _train_leg(*sys.argv[2:])
