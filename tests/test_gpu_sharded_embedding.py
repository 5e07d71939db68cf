"""A learned node-feature table sharded by rows with its Adam moments (``dist.ShardedEmbedding``), on one B200:

* the row-range table walk (grapes_adam_embed_rows, grapes_embed_merge_adam_rows) over W = 1, 2, 3, 8 ranges equals the
  whole-table walk bit for bit, and never touches a shard buffer behind its rows (NaN canaries);
* the table epoch (grapes_embed_epoch_post / _wait) for a world of one and two emulated peers on one device;
* engines over W emulated shards against the replicated learned-table engine: a recorded step, three Adam steps eager
  and from a graph, predict and full-batch evaluation, all bit for bit; and train() with one process.

Deliberate errors and the test that catches each: the walk started at row0 + 1, or the merge's walk over the whole
table instead of the range -> test_row_range_walk_equals_whole_table / test_merge_rows_equal_whole_table_merge (both
also check in place that a shifted or foreign range is seen)."""
import ctypes

import pytest
import torch

from test_gpu_embed import _bitmap
from test_gpu_embed_dp_kernels import _ctx, _merge, _merge_args, _slots

pytestmark = pytest.mark.gpu

GO_FAIL = -(1 << 31)                      # 0x80000000 as int32
LR = 1e-2


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _same(a, b, where=""):
    """Bit-identical nested records (NaN included)."""
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
        assert torch.equal(_bits(a.contiguous()), _bits(b.contiguous())), where
    else:
        assert a == b or (a != a and b != b), f"{where}: {a} != {b}"


def _start(N, F, gen, dev):
    """A table, and moments that are non-zero on every third row (rows touched earlier, moved by their moments alone)."""
    x = torch.randn(N, F, generator=gen)
    m, v = torch.zeros(N, F), torch.zeros(N, F)
    m[::3] = torch.randn(m[::3].shape, generator=gen) * 1e-2
    v[::3] = torch.rand(v[::3].shape, generator=gen) * 1e-3
    return [t.to(dev) for t in (x, m, v)]


def _split(tabs, bounds):
    """Per range: three buffers of (max rows + 2) rows, the range's rows at the top, NaN behind them."""
    W = len(bounds) - 1
    rows = max(bounds[r + 1] - bounds[r] for r in range(W))
    out = []
    for r in range(W):
        lo, hi = bounds[r], bounds[r + 1]
        bufs = []
        for t in tabs:
            b = torch.full((rows + 2, t.shape[1]), float("nan"), device=t.device)
            b[:hi - lo] = t[lo:hi]
            bufs.append(b)
        out.append(bufs)
    return out


def _check_shards(shards, bounds, want, where):
    for r, bufs in enumerate(shards):
        lo, hi = bounds[r], bounds[r + 1]
        for b in bufs:
            assert b[hi - lo:].isnan().all(), f"{where}: range {r} wrote behind its rows"
    for i in range(3):
        _same(torch.cat([bufs[i][:bounds[r + 1] - bounds[r]] for r, bufs in enumerate(shards)]), want[i], where)


@pytest.mark.parametrize("N", [1003, 10])
def test_row_range_walk_equals_whole_table(cuda_device, N):
    """grapes_adam_embed_rows over every range of W = 1, 2, 3, 8 (N = 10: empty last ranges) = grapes_adam_embed,
    three steps with different row sets, gradient pitch > F; rows never touched and rows moved by their moments only."""
    from grapes_b200._lib import lib
    from grapes_b200.dist import feature_bounds
    dev, L = cuda_device, lib()
    F, ldg = 16, 24
    g = _ctx(N, dev)
    st = torch.cuda.current_stream().cuda_stream
    for W in (1, 2, 3, 8):
        gen = torch.Generator().manual_seed(W)
        whole = _start(N, F, gen, dev)
        bounds = feature_bounds(N, W)
        shards = _split(whole, bounds)
        steps = torch.zeros(2, device=dev)
        for it in range(3):
            ids = torch.sort(torch.randperm(N, generator=gen)[:max(1, N // 5)]).values
            grows = torch.randn(ids.numel(), ldg, generator=gen).to(dev)
            bm, pref = _bitmap(ids, N, dev)
            args = (F, bm.data_ptr(), pref.data_ptr(), grows.data_ptr(), ldg, LR, 0.9, 0.999, 1e-8, steps.data_ptr(), st)
            wrong = [[b.clone() for b in bufs] for bufs in shards] if W == 3 and it == 0 else None
            L.grapes_adam_embed(g.ctx, *[t.data_ptr() for t in whole], N, *args)
            for r, bufs in enumerate(shards):
                L.grapes_adam_embed_rows(g.ctx, *[b.data_ptr() for b in bufs], N, bounds[r], bounds[r + 1] - bounds[r],
                                         *args)
            if wrong is not None:
                # the check sees a walk that starts one row late
                for r, bufs in enumerate(wrong):
                    n = bounds[r + 1] - bounds[r]
                    L.grapes_adam_embed_rows(g.ctx, *[b.data_ptr() for b in bufs], N, min(bounds[r] + 1, N - n), n,
                                             *args)
                with pytest.raises(AssertionError):
                    _check_shards(wrong, bounds, whole, "shifted")
            steps[0] += 1
            torch.cuda.synchronize()
            _check_shards(shards, bounds, whole, f"N {N} W {W} step {it}")


def test_merge_rows_equal_whole_table_merge(cuda_device):
    """grapes_embed_merge_adam_rows over every range of W = 1, 2, 3, 8 on hand-built slots of three ranks =
    grapes_embed_merge_adam over the whole table; a go word carrying GO_FAIL makes the launch a no-op."""
    from grapes_b200._lib import lib
    from grapes_b200.dist import feature_bounds
    dev, L = cuda_device, lib()
    N, F, cap, world = 1000, 16, 96, 3
    g = _ctx(N, dev)
    st = torch.cuda.current_stream().cuda_stream

    def merge_rows(slots, state, bufs, row0, rows, steps):
        a = _merge_args(N, F, world * cap, dev)
        L.grapes_embed_merge_adam_rows(g.ctx, slots.data_ptr(), world, cap, F, state, a["bm"].data_ptr(),
                                       a["pref"].data_ptr(), a["ids"].data_ptr(), a["ids"].numel(), a["cnt"].data_ptr(),
                                       a["mean"].data_ptr(), *[b.data_ptr() for b in bufs], N, row0, rows, LR, 0.9,
                                       0.999, 1e-8, steps.data_ptr(), a["ovf"].data_ptr(), st)
        return a

    for W in (1, 2, 3, 8):
        gen = torch.Generator().manual_seed(10 + W)
        whole = _start(N, F, gen, dev)
        bounds = feature_bounds(N, W)
        shards = _split(whole, bounds)
        steps = torch.zeros(2, device=dev)
        for it in range(3):
            payloads = []
            for r in range(world):
                k = int(torch.randint(1, cap + 1, (1,), generator=gen))
                ids = torch.sort(torch.randperm(N, generator=gen)[:k]).values
                payloads.append((ids, torch.randn(ids.numel(), F, generator=gen)))
            slots = _slots(payloads, cap, F)[0].to(dev)
            steps[0] += 1
            wrong = [[b.clone() for b in bufs] for bufs in shards] if W == 2 and it == 0 else None
            _merge(L, g, slots, world, cap, F, None, _merge_args(N, F, world * cap, dev), *whole, N, LR, steps)
            for r, bufs in enumerate(shards):
                merge_rows(slots, None, bufs, bounds[r], bounds[r + 1] - bounds[r], steps)
            if wrong is not None:
                # the check sees a merge whose walk ignores the range (here: range 0's buffers walked over range 1's rows)
                merge_rows(slots, None, wrong[1], bounds[1], bounds[2] - bounds[1], steps)
                merge_rows(slots, None, wrong[0], bounds[1], bounds[2] - bounds[1], steps)
                with pytest.raises(AssertionError):
                    _check_shards(wrong, bounds, whole, "foreign range")
            torch.cuda.synchronize()
            _check_shards(shards, bounds, whole, f"W {W} step {it}")
    # go word with GO_FAIL (slots read through the state: parity of the go word): nothing moves, canaries included
    state = torch.zeros(int(L.cdll.grapes_peer_state_words()), dtype=torch.int32, device=dev)
    state[4] = GO_FAIL | 1
    two = torch.cat([slots, slots])
    before = [[b.clone() for b in bufs] for bufs in shards]
    for r, bufs in enumerate(shards):
        merge_rows(two, state.data_ptr(), bufs, bounds[r], bounds[r + 1] - bounds[r], steps)
    torch.cuda.synchronize()
    _same(before, shards, "GO_FAIL")


def _epoch(L, world, dev):
    words = int(L.cdll.grapes_embed_epoch_words(world))
    bufs = [torch.zeros(words, dtype=torch.int32, device=dev) for _ in range(world)]
    return bufs, (ctypes.c_void_p * world)(*[b.data_ptr() for b in bufs])


def test_epoch_post_and_wait(cuda_device):
    """World of one; two emulated peers (two buffers, a host array of their pointers): a post advances the words, a
    wait with everyone posted passes, a word left behind times out with GRAPES_OVF_PEER_TIMEOUT (and the sticky
    failure of a state) and the launch returns; a post under GO_FAIL does nothing; a captured post replayed three
    times advances the count by three."""
    from grapes_b200._lib import lib
    dev, L = cuda_device, lib()
    g = _ctx(64, dev)
    st = torch.cuda.current_stream().cuda_stream
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    # world of one
    bufs, ptrs = _epoch(L, 1, dev)
    L.grapes_embed_epoch_post(g.ctx, ptrs, 0, 1, None, st)
    L.grapes_embed_epoch_wait(g.ctx, bufs[0].data_ptr(), 1, None, err.data_ptr(), 1000, st)
    torch.cuda.synchronize()
    assert bufs[0].tolist() == [1, 1] and int(err.item()) == 0
    # two peers
    bufs, ptrs = _epoch(L, 2, dev)
    state = torch.zeros(int(L.cdll.grapes_peer_state_words()), dtype=torch.int32, device=dev)
    L.grapes_embed_epoch_post(g.ctx, ptrs, 0, 2, state.data_ptr(), st)
    torch.cuda.synchronize()
    assert bufs[0].tolist() == [1, 0, 1] and bufs[1].tolist() == [1, 0, 0]
    L.grapes_embed_epoch_wait(g.ctx, bufs[0].data_ptr(), 2, state.data_ptr(), err.data_ptr(), 2000, st)
    torch.cuda.synchronize()                       # rank 1 has not posted: bounded spin, flagged, sticky failure
    assert int(err.item()) & 32 and int(state[3].item()) == 1
    err.zero_()
    L.grapes_embed_epoch_wait(g.ctx, bufs[1].data_ptr(), 2, None, err.data_ptr(), 2000, st)
    L.grapes_embed_epoch_post(g.ctx, ptrs, 1, 2, None, st)
    torch.cuda.synchronize()                       # rank 1 at count 0 passes; its post reaches both buffers
    assert int(err.item()) == 0
    assert bufs[0].tolist() == [1, 1, 1] and bufs[1].tolist() == [1, 1, 1]
    for r in range(2):
        L.grapes_embed_epoch_wait(g.ctx, bufs[r].data_ptr(), 2, None, err.data_ptr(), 2000, st)
    torch.cuda.synchronize()
    assert int(err.item()) == 0
    # a failed step posts nothing
    state.zero_()
    state[4] = GO_FAIL | 2
    L.grapes_embed_epoch_post(g.ctx, ptrs, 0, 2, state.data_ptr(), st)
    torch.cuda.synchronize()
    assert bufs[0].tolist() == [1, 1, 1] and bufs[1].tolist() == [1, 1, 1]
    # graph replay advances the device count
    bufs, ptrs = _epoch(L, 1, dev)
    torch.cuda.synchronize()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        L.grapes_embed_epoch_post(g.ctx, ptrs, 0, 1, None, torch.cuda.current_stream().cuda_stream)
    for _ in range(3):
        gr.replay()
    torch.cuda.synchronize()
    assert bufs[0].tolist() == [3, 3]


def _engines(dev, W, multilabel=False, F=64, **kw):
    from grapes_b200.dist import ShardedEmbedding
    from grapes_b200.engine import GrapesEngine
    from grapes_b200.graph import DeviceGraph
    from grapes_b200.synth import SHAPES, make_synth
    cfg = dict(SHAPES["small"])
    d = make_synth("small", seed=3, multilabel=multilabel)
    x = torch.empty(d.num_nodes, F).normal_(generator=torch.Generator().manual_seed(4))
    g = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=dev)
    shards = ShardedEmbedding.emulate(x.to(dev), W)
    for s in shards:                                        # NaN behind every shard's rows
        s.table.rows[s.hi - s.lo:] = float("nan")
    hp = dict(num_classes=d.num_classes, batch_size=cfg["batch_size"], num_samples=cfg["num_samples"],
              sampling_hops=cfg["sampling_hops"], hidden_dim=256, seed=5, embed_nodes=True)
    hp.update(kw)
    rep = GrapesEngine(g, x.to(dev), d.y.to(dev), **hp)
    sh = GrapesEngine(g, shards[W - 1], d.y.to(dev), **hp)
    assert sh.x is None and sh.embed_shards is shards[W - 1]
    d.x = x
    return d, rep, sh, shards


def _check_table(rep, sh, where):
    es = sh.embed_shards
    _same(rep.params, sh.params, f"{where} params")
    _same(rep.x, es.to_dense(), f"{where} table")
    m, v = es.moments_dense()
    _same(rep.emb_exp_avg, m, f"{where} exp_avg")
    _same(rep.emb_exp_avg_sq, v, f"{where} exp_avg_sq")
    for s in es.shards:
        assert s.table.rows[s.hi - s.lo:].isnan().all(), where


@pytest.mark.parametrize("case", ["tb", "reinforce", "multilabel", "dropout", "simt", "wide"])
def test_step_equals_replicated_learned_table(cuda_device, case):
    kw = {"tb": {}, "reinforce": dict(reinforce_baseline=True), "multilabel": dict(multilabel=True),
          "dropout": dict(dropout=0.3), "simt": dict(use_tensor_cores=False), "wide": {}}[case]
    for W in (1, 2, 3, 8):
        d, rep, sh, _ = _engines(cuda_device, W, **kw)
        if case == "wide":                                  # the relabel + build_csr classifier form
            rep.PREP_MAX_ROWS = sh.PREP_MAX_ROWS = 64
            assert rep.cap_A > 64
        t = d.train_mask.nonzero().squeeze(1)[:rep.B].to(torch.int32).to(cuda_device)
        _same(rep.step(t, apply_optim=False, record=True), sh.step(t, apply_optim=False, record=True), f"{case} W {W}")
        _same(rep.step(t, record=True), sh.step(t, record=True), f"{case} W {W} with Adam")
        _check_table(rep, sh, f"{case} W {W}")
        rep.check_overflow(); sh.check_overflow()


@pytest.mark.parametrize("W", [1, 2, 3, 8])
def test_adam_steps_graph_replay_predict_and_full_batch_eval(cuda_device, W):
    """Three Adam steps eager, three replayed from a graph, then predict and full-batch evaluation over the shards."""
    from grapes_b200 import eval as E
    from grapes_b200 import train as T
    from grapes_b200.gcn import GCN, LocalRowTable, ShardedGraphNorm, sharded_layer1, sharded_layer2
    dev = cuda_device
    d, rep, sh, shards = _engines(dev, W)
    idx = d.train_mask.nonzero().squeeze(1).to(torch.int32).to(dev)
    batches = [b.contiguous() for b in torch.split(idx, rep.B)][:6]
    for i in range(3):
        for eng in (rep, sh):
            eng.step(batches[i])
        torch.cuda.synchronize()
        _check_table(rep, sh, f"W {W} eager step {i}")
    for i in range(3, 6):
        for eng in (rep, sh):
            eng.step(batches[i], use_graph=True, next_targets=batches[i + 1] if i + 1 < 6 else None)
            eng.check_overflow()
    _check_table(rep, sh, f"W {W} graph")
    test = d.test_mask.nonzero().squeeze(1).to(torch.int32).to(dev)[:rep.B].contiguous()
    preds = []
    for eng in (rep, sh):
        out = torch.zeros(rep.B, dtype=torch.int32, device=dev)
        eng.predict(test, out)
        eng.check_overflow()
        preds.append(out)
    _same(preds[0], preds[1], "predict")
    # full-batch evaluation: the replicated one-process evaluate() against the row-partitioned forward over the shards
    mask = d.test_mask.to(dev)
    y = d.y.to(dev)
    d.x = rep.x
    want = T.evaluate(rep, d, mask, full_batch=True)
    gcn_c = GCN(sh.F, [sh.D, sh.C]).to(dev).eval()
    gcn_c.load_state_dict(sh.state_dicts()["gcn_c"])
    ei = d.edge_index.to(dev)
    parts = [ShardedGraphNorm(sh.g, W, r, edge_index=ei) for r in range(W)]
    ztabs = LocalRowTable.make(W, max(p.rows for p in parts), (sh.C + 3) // 4 * 4, dev)
    for p in parts:
        sharded_layer1(gcn_c, shards[p.rank], p, ztabs[p.rank], slab_rows=97)
    counts = torch.zeros(3, dtype=torch.int64, device=dev)
    for p in parts:
        counts += sharded_layer2(gcn_c, p, ztabs[p.rank], y=y, mask=mask)[1]
    got = (E._mean_of_hits(int(counts[0]), int(counts[1])),) * 2
    assert got == want, (W, got, want)


def test_train_one_process_ignores_shard_embeddings(cuda_device):
    from grapes_b200 import train as T
    from grapes_b200.args import Arguments
    from grapes_b200.synth import make_synth
    f1s = []
    for shard in (False, True):
        a = Arguments()
        a.dataset, a.max_epochs, a.batch_size, a.num_samples, a.sampling_hops = "small", 2, 128, 32, 3
        a.embed_nodes, a.node_emb_dim, a.eval_frequency = True, 32, 1
        f1, *_ = T.train(a, data=make_synth("small", seed=2), device=cuda_device, shard_embeddings=shard)
        assert T.train.last_engine.embed_shards is None
        f1s.append(f1)
    assert f1s[0] == f1s[1]
