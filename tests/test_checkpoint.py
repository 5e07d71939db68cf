"""Checkpoint format and protocol on the CPU (``grapes_b200.checkpoint``): the row-offset table writer and its
memory-mapped reader across world sizes, the atomicity of a save that dies, the size / CRC and ``meta.json`` checks,
save / load of the host-side state and the parameter-checksum agreement under gloo with two ranks, and the per-run
directories of ``python -m grapes_b200.main`` with ``GRAPES_CHECKPOINT_DIR``.  The engine is a CPU stand-in with the
attributes a checkpoint reads and writes."""
import json
import os
import socket
import warnings

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from grapes_b200 import checkpoint as C
from grapes_b200._lib import GrapesError
from grapes_b200.args import Arguments
from grapes_b200.dist import feature_bounds


class _Stub:
    """What save() / load() touch of a GrapesEngine, on the CPU."""

    def __init__(self, seed=0, N=37, F=8, embed=False, world=1):
        g = torch.Generator().manual_seed(seed)
        self.N, self.F, self.C, self.D, self.H, self.k, self.B = N, F, 3, 16, 2, 4, 8
        self.n_par = 30
        self.x_bf16, self.embed_nodes, self.multilabel = False, embed, False
        self.dp_world, self.dp_group, self.peer, self.features, self.embed_shards = world, None, None, None, None
        self.device = torch.device("cpu")
        self.params = torch.randn(self.n_par, generator=g)
        self.exp_avg, self.exp_avg_sq = torch.randn(self.n_par, generator=g), torch.rand(self.n_par, generator=g)
        self.adam_steps = torch.tensor([float(seed + 3)] * 2)
        self.rng_state = torch.tensor([seed, 100 + seed], dtype=torch.int64)
        self.drop_state = torch.tensor([seed, 200 + seed], dtype=torch.int64)
        self.overflow = torch.zeros(1, dtype=torch.int32)
        self.scal = torch.zeros(16)
        if embed:
            self.x, self.emb_exp_avg = torch.randn(N, F, generator=g), torch.randn(N, F, generator=g)
            self.emb_exp_avg_sq = torch.rand(N, F, generator=g)
        self._front_ready, self._pref_key = [True, False], (1, 2)

    def _views(self):
        return {"gcn_c": {"w": self.params[:10]}, "gcn_gf": {"w": self.params[10:22]}, "gcn_z": {"w": self.params[22:]}}

    def state_dicts(self):
        return self._views()

    def load_state_dicts(self, **sds):
        for k, v in self._views().items():
            v["w"].copy_(sds[k]["w"])

    def tensors(self):
        names = ["params", "exp_avg", "exp_avg_sq", "adam_steps", "rng_state", "drop_state"]
        if self.embed_nodes:
            names += ["x", "emb_exp_avg", "emb_exp_avg_sq"]
        return {n: getattr(self, n) for n in names}


def _same_state(a, b):
    ta, tb = a.tensors(), b.tensors()
    for n in ta:
        assert torch.equal(ta[n], tb[n]), n


@pytest.mark.parametrize("N", [1003, 10, 2])
def test_row_writer_round_trip_across_world_sizes(tmp_path, N):
    """A [N, F] table written by W = 1, 2, 3, 8 owners at their row offsets (chunks of 3 rows) reads back bit-identically,
    whole and through the rows of W' = 1, 3, 8 readers; N = 2 leaves ranges empty."""
    F = 12
    want = torch.randn(N, F, generator=torch.Generator().manual_seed(N))
    want[0, 0] = float("nan")
    for W in (1, 2, 3, 8):
        path = str(tmp_path / f"t{W}.f32")
        b = feature_bounds(N, W)
        for r in reversed(range(W)):                     # any order: every owner extends the file to its full size
            C.write_rows(path, want[b[r]:b[r + 1]], b[r], N, chunk_bytes=3 * 4 * F)
        assert os.path.getsize(path) == 4 * N * F
        got = C.read_rows(path, N, F)
        assert torch.equal(got.view(torch.int32), want.view(torch.int32)), W
        for W2 in (1, 3, 8):
            b2 = feature_bounds(N, W2)
            parts = torch.cat([got[b2[r]:b2[r + 1]].clone() for r in range(W2)])
            assert torch.equal(parts.view(torch.int32), want.view(torch.int32)), (W, W2)


def test_save_load_round_trip_and_in_place(tmp_path):
    src, dst = _Stub(seed=1, embed=True), _Stub(seed=2, embed=True)
    before = {n: t.data_ptr() for n, t in dst.tensors().items()}
    path = C.save(src, str(tmp_path), dict(epoch=2, batch=5, step=17, acc_c=0.5, acc_gfn=1.5, last={"a": 1.0}),
                  args=Arguments())
    assert os.path.basename(path) == "step-000000017" and C.latest(str(tmp_path)) == path
    assert sorted(os.listdir(path)) == sorted(["meta.json", "model.pt", "optim.pt", "rank0.pt", *C.TABLE_FILES])
    loop = C.load(dst, str(tmp_path), args=Arguments())
    _same_state(src, dst)
    assert {n: t.data_ptr() for n, t in dst.tensors().items()} == before          # nothing rebound
    assert dst._front_ready == [False, False] and dst._pref_key is None
    assert loop == dict(epoch=2, batch=5, step=17, acc_c=0.5, acc_gfn=1.5, last={"a": 1.0})
    t, m, v = C.table_source(path)
    assert torch.equal(t, src.x) and torch.equal(m, src.emb_exp_avg) and torch.equal(v, src.emb_exp_avg_sq)
    meta = C.read_meta(path)
    assert meta["sizes"]["table.f32"] == 4 * src.N * src.F and "table.f32" not in meta["crc"]
    assert meta["args"] == Arguments().as_dict() and meta["step"] == 17


def test_keeps_two_newest_checkpoints(tmp_path):
    s = _Stub()
    for step in (1, 2, 3, 4):
        C.save(s, str(tmp_path), dict(step=step))
    names = sorted(n for n in os.listdir(tmp_path) if n.startswith("step-"))
    assert names == ["step-000000003", "step-000000004"]
    with open(tmp_path / "LATEST") as f:
        assert f.read().strip() == "step-000000004"
    C.save(s, str(tmp_path), dict(step=4, epoch=9))    # the same step again replaces it
    assert C.read_meta(str(tmp_path))["epoch"] == 9


@pytest.mark.parametrize("where", ["before_meta", "before_latest"])
def test_a_save_that_dies_leaves_the_previous_checkpoint(tmp_path, monkeypatch, where):
    old, new = _Stub(seed=1, embed=True), _Stub(seed=2, embed=True)
    C.save(old, str(tmp_path), dict(step=1))

    def boom(*a, **k):
        raise RuntimeError("process died")
    if where == "before_meta":
        monkeypatch.setattr(C, "_commit", boom)
    else:
        monkeypatch.setattr(os, "replace", boom)
    with pytest.raises(RuntimeError):
        C.save(new, str(tmp_path), dict(step=2))
    monkeypatch.undo()
    assert C.latest(str(tmp_path)).endswith("step-000000001")
    got = _Stub(seed=3, embed=True)
    assert C.load(got, str(tmp_path))["step"] == 1
    _same_state(old, got)
    C.save(new, str(tmp_path), dict(step=2))           # the next save cleans up and succeeds
    assert C.latest(str(tmp_path)).endswith("step-000000002")
    assert not any(n.endswith(".tmp") for n in os.listdir(tmp_path))


def test_size_and_crc_checks(tmp_path):
    s = _Stub(embed=True)
    path = C.save(s, str(tmp_path), dict(step=1))
    with open(os.path.join(path, "table_m.f32"), "r+b") as f:
        f.truncate(4 * s.N * s.F - 4)
    with pytest.raises(GrapesError, match="table_m.f32"):
        C.load(_Stub(embed=True), path)
    path = C.save(s, str(tmp_path), dict(step=2))
    p = os.path.join(path, "model.pt")
    raw = bytearray(open(p, "rb").read())
    raw[len(raw) // 2] ^= 1
    open(p, "wb").write(bytes(raw))
    with pytest.raises(GrapesError, match="model.pt.*CRC"):
        C.load(_Stub(embed=True), path)


def test_save_refusals(tmp_path):
    s = _Stub()
    s.overflow[0] = 2
    with pytest.raises(GrapesError, match="flag word"):
        C.save(s, str(tmp_path), dict(step=1))
    s.overflow[0] = 0
    s.scal[15] = 32.
    with pytest.raises(GrapesError, match="flag word"):
        C.save(s, str(tmp_path), dict(step=1))
    s.scal[15] = 0.
    os.makedirs(C.step_path(str(tmp_path), 5))
    with pytest.raises(GrapesError, match="not a checkpoint"):
        C.save(s, str(tmp_path), dict(step=5))


def test_meta_validation(tmp_path):
    s = _Stub(embed=True)
    meta = C.read_meta(C.save(s, str(tmp_path), dict(step=1), args=Arguments()))
    cur = C.describe(s)
    for key in C.SHAPE_FIELDS:
        bad = dict(meta)
        bad[key] = "other"
        with pytest.raises(GrapesError, match=key):
            C.check_meta(bad, cur)
    with pytest.raises(GrapesError, match="format"):
        C.check_meta(dict(meta, format=99), cur)
    for key, val in (("hidden_dim", 128), ("lr_gc", 0.5), ("dropout", 0.5), ("seed", 3), ("random_sampling", True)):
        a = Arguments()
        setattr(a, key, val)
        with pytest.raises(GrapesError, match=key):
            C.check_meta(meta, cur, a)
    a = Arguments()
    a.max_epochs, a.eval_frequency, a.runs, a.notes = 99, 1, 3, "resumed"
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        C.check_meta(meta, cur, a)                    # allowed, silently
    with pytest.warns(UserWarning, match="world 1 -> 2"):
        C.check_meta(meta, dict(cur, world=2), a)
    with pytest.warns(UserWarning, match="shard_embeddings"):
        C.check_meta(meta, dict(cur, shard_embeddings=True), a)
    # through load(): the error names the field
    small = _Stub(embed=True, F=4)
    with pytest.raises(GrapesError, match="F = 8"):
        C.load(small, str(tmp_path))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, root, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    g = dist.group.WORLD
    s = _Stub(seed=4, embed=True, world=world)
    s.rng_state[1] += rank                            # per-rank host-side state
    path = C.save(s, root, dict(epoch=1, batch=3, step=6, acc_c=float(rank), acc_gfn=2.0 + rank, last={"r": rank}),
                  group=g)
    got = _Stub(seed=9, embed=True, world=world)
    loop = C.load(got, root, group=g)
    res = dict(path=path, loop=loop, same=all(torch.equal(got.tensors()[n], s.tensors()[n]) for n in s.tensors()))
    s.params[3] += float(rank)                        # rank 1's parameters differ
    try:
        C.save(s, root, dict(step=7), group=g)
        res["refused"] = None
    except GrapesError as exc:
        res["refused"] = str(exc)
    res["latest"] = C.latest(root)
    out[rank] = res
    dist.barrier()
    dist.destroy_process_group()


def test_gloo_two_ranks_save_load_and_parameter_agreement(tmp_path):
    world, root = 2, str(tmp_path)
    out = mp.Manager().dict()
    mp.spawn(_worker, args=(world, _free_port(), root, out), nprocs=world, join=True)
    for r in range(world):
        o = out[r]
        assert o["same"], r
        assert o["loop"] == dict(epoch=1, batch=3, step=6, acc_c=float(r), acc_gfn=2.0 + r, last={"r": r})
        assert o["refused"] is not None and "parameters differ" in o["refused"], o["refused"]
        assert o["latest"] == o["path"]
    assert sorted(os.listdir(out[0]["path"])) == sorted(["meta.json", "model.pt", "optim.pt", "rank0.pt", "rank1.pt",
                                                         *C.TABLE_FILES])
    assert C.read_meta(root)["world"] == 2


def test_main_checkpoint_dir_per_run(tmp_path, monkeypatch):
    from grapes_b200 import main as M
    calls = []

    def fake_train(args, **kw):
        calls.append(kw)
        return 0.5, [1.0], [1.0], [1.0]
    monkeypatch.setattr(M, "train", fake_train)
    monkeypatch.setenv("GRAPES_CHECKPOINT_DIR", str(tmp_path))
    M.main(["--runs", "3", "--max_epochs", "1"])
    assert calls == [dict(checkpoint_dir=os.path.join(str(tmp_path), f"run{r}"), resume=True) for r in range(3)]
    monkeypatch.delenv("GRAPES_CHECKPOINT_DIR")
    calls.clear()
    M.main(["--runs", "2"])
    assert calls == [{}, {}]


def test_train_checkpoint_arguments():
    from grapes_b200.train import train
    for kw in (dict(checkpoint_every=5), dict(resume=True), dict(checkpoint_dir="d", checkpoint_every=-1)):
        with pytest.raises(GrapesError, match="checkpoint_dir"):
            train(Arguments(), **kw)


def test_meta_is_plain_json(tmp_path):
    path = C.save(_Stub(), str(tmp_path), dict(step=3, epoch=1, batch=2), args=Arguments())
    with open(os.path.join(path, "meta.json")) as f:
        meta = json.load(f)
    for key in ("format", "world", "exchange", "shard_features", "shard_embeddings", "args", "N", "F", "C", "D", "H",
                "k", "B", "dtype", "embed_nodes", "multilabel", "epoch", "batch", "step", "sizes", "crc"):
        assert key in meta, key
    assert set(meta["crc"]) == {"model.pt", "optim.pt", "rank0.pt"}
