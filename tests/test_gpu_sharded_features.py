"""A feature table sharded by rows across data-parallel ranks, on one B200 with W emulated ranks (W allocations of this
device, which is all the peer kernels see): the peer gathers (grapes_aggregate_peer, grapes_aggregate_rows64_peer_x)
against the replicated ones, a training step / predict / full-batch evaluation over the sharded table against the
replicated engine and evaluate(), all bit for bit, and the refusals.

Every shard allocation holds N + 1 rows, NaN outside the shard's own rows and in its pad columns, so a wrong owner or row
offset reads a NaN canary instead of memory outside the allocation.  Deliberate errors in k_agg_px and the test that
catches each: `>` for `>=` in the owner select, an unshifted row for the last shard, and a dropped self term ->
test_hop_form_bit_identical / test_slab_form_bit_identical; indicator bits read by global id ->
test_hop_form_bit_identical (num_ind > 0, ind_bits defined for every global id)."""
import ctypes

import pytest
import torch

pytestmark = pytest.mark.gpu


def _bits(t):
    return t.view(torch.int16 if t.element_size() == 2 else torch.int32) if t.is_floating_point() else t


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


def _shards(x, W, ldx):
    """W allocations of N + 1 rows each: shard o's rows at the top, NaN everywhere else (rows and pad columns)."""
    from grapes_b200.dist import feature_bounds
    N, F = x.shape
    bounds = feature_bounds(N, W)
    tabs = []
    for o in range(W):
        t = torch.full((N + 1, ldx), float("nan"), dtype=x.dtype, device=x.device)
        t[:bounds[o + 1] - bounds[o], :F] = x[bounds[o]:bounds[o + 1]]
        tabs.append(t)
    ptrs = (ctypes.c_void_p * W)(*[t.data_ptr() for t in tabs])
    return tabs, ptrs, (ctypes.c_int64 * (W + 1))(*bounds)


def _local_graph(N, n, cap_n, dev, gen):
    """A hop-shaped local structure: n rows of cap_n, node ids `nodes` (distinct global ids), sources ascending per row,
    rows 0 and 1 with 40 and 1500 sources (past one and 32 warp-wide loads), dinv in (0.1, 1]."""
    nodes = torch.randperm(N, generator=gen)[:cap_n].to(torch.int32)
    deg = torch.randint(0, 12, (n,), generator=gen)
    deg[0], deg[1] = 40, 1500
    deg = deg.clamp(max=n)
    src = [torch.sort(torch.randperm(n, generator=gen)[:int(d)]).values for d in deg]
    in_off = torch.zeros(cap_n + 1, dtype=torch.int32)
    in_off[1:n + 1] = torch.cumsum(deg, 0).to(torch.int32)
    in_off[n + 1:] = in_off[n]
    in_src = torch.cat(src).to(torch.int32)
    dinv = torch.rand(cap_n, generator=gen) * 0.9 + 0.1
    ind_bits = torch.randint(0, 1 << 30, (max(N, cap_n),), generator=gen).to(torch.int32)
    return [t.to(dev) for t in (nodes, in_off, in_src, dinv, ind_bits)]


CASES = [(2, torch.float32), (3, torch.float32), (36, torch.float32), (100, torch.float32), (602, torch.float32),
         (1433, torch.float32), (128, torch.bfloat16), (130, torch.bfloat16)]


@pytest.mark.parametrize("F,dtype", CASES)
def test_hop_form_bit_identical(cuda_device, F, dtype):
    """grapes_aggregate_peer = grapes_aggregate / grapes_aggregate_bf16 over the whole table: W in {1, 2, 3, 8}, num_ind in
    {0, 3, 8}, out or the hi / lo split with ones_col, bias + relu, n_dev < cap_n, hub rows of 40 and 1500 sources."""
    from grapes_b200._lib import lib
    from grapes_b200.graph import DeviceGraph
    dev = cuda_device
    L = lib()
    holder = DeviceGraph.from_edge_index(torch.tensor([[0], [1]]), 2, device=dev)      # owns the library context
    ctx = holder.ctx
    gen = torch.Generator().manual_seed(F)
    N, n, cap_n = 6000, 2500, 3000
    x = torch.randn((N, F), generator=gen).to(dev, dtype)
    ldx = (F + 3) // 4 * 4
    xr = torch.zeros((N, ldx), dtype=dtype, device=dev)
    xr[:, :F] = x
    nodes, in_off, in_src, dinv, ind_bits = _local_graph(N, n, cap_n, dev, gen)
    n_dev = torch.tensor([n], dtype=torch.int32, device=dev)
    bias = torch.randn(F, generator=gen).to(dev)
    agg = L.grapes_aggregate_bf16 if dtype == torch.bfloat16 else L.grapes_aggregate
    st = torch.cuda.current_stream().cuda_stream
    for W in (1, 2, 3, 8):
        tabs, ptrs, bounds = _shards(x, W, ldx)
        for num_ind in (0, 3, 8):
            for split in (False, True):
                for b, relu in ((None, 0), (bias, 1)):
                    ldo = (F + num_ind + 1 + 3) // 4 * 4
                    ones = F + num_ind if split else -1
                    outs = []
                    for peer in (False, True):
                        o = [torch.full((cap_n + 1, ldo), float("nan"), device=dev) for _ in range(3)]
                        out, hi, lo = (None, o[1], o[2]) if split else (o[0], None, None)
                        args = (nodes.data_ptr(), n_dev.data_ptr(), cap_n, in_off.data_ptr(), in_src.data_ptr(),
                                dinv.data_ptr(), ind_bits.data_ptr() if num_ind else None, num_ind,
                                None if b is None else b.data_ptr(), relu,
                                None if out is None else out.data_ptr(), ldo, None if hi is None else hi.data_ptr(),
                                None if lo is None else lo.data_ptr(), ones, st)
                        if peer:
                            L.grapes_aggregate_peer(ctx, ptrs, bounds, W, int(dtype == torch.bfloat16), F, ldx, *args)
                        else:
                            agg(ctx, xr.data_ptr(), F, ldx, *args)
                        outs.append(o)
                    torch.cuda.synchronize()
                    assert not outs[1][1 if split else 0][:n, :F].isnan().any()
                    _same(outs[0], outs[1], f"W {W} num_ind {num_ind} split {split} relu {relu}")


def test_hop_form_more_ranks_than_rows(cuda_device):
    """N < W: empty shards (NULL bases) are never selected."""
    from grapes_b200._lib import lib
    from grapes_b200.graph import DeviceGraph
    dev = cuda_device
    L = lib()
    holder = DeviceGraph.from_edge_index(torch.tensor([[0], [1]]), 2, device=dev)      # owns the library context
    ctx = holder.ctx
    x = torch.randn((3, 8), device=dev)
    nodes = torch.tensor([2, 0, 1], dtype=torch.int32, device=dev)
    in_off = torch.tensor([0, 2, 3, 3], dtype=torch.int32, device=dev)
    in_src = torch.tensor([1, 2, 0], dtype=torch.int32, device=dev)
    dinv = torch.tensor([0.5, 0.7, 0.9], device=dev)
    n_dev = torch.tensor([3], dtype=torch.int32, device=dev)
    ref = torch.full((3, 8), float("nan"), device=dev)
    L.grapes_aggregate(ctx, x.data_ptr(), 8, 8, nodes.data_ptr(), n_dev.data_ptr(), 3, in_off.data_ptr(),
                       in_src.data_ptr(), dinv.data_ptr(), None, 0, None, 0, ref.data_ptr(), 8, None, None, -1,
                       torch.cuda.current_stream().cuda_stream)
    tabs, ptrs, bounds = _shards(x, 8, 8)
    assert list(bounds) == [0, 1, 2, 3, 3, 3, 3, 3, 3]
    for o in range(3, 8):
        ptrs[o] = None
    got = torch.full((3, 8), float("nan"), device=dev)
    L.grapes_aggregate_peer(ctx, ptrs, bounds, 8, 0, 8, 8, nodes.data_ptr(), n_dev.data_ptr(), 3, in_off.data_ptr(),
                            in_src.data_ptr(), dinv.data_ptr(), None, 0, None, 0, got.data_ptr(), 8, None, None, -1,
                            torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    _same(ref, got)


@pytest.mark.parametrize("F,dtype", [(3, torch.float32), (6, torch.float32), (36, torch.float32),
                                     (128, torch.bfloat16), (130, torch.bfloat16)])
def test_slab_form_bit_identical(cuda_device, F, dtype):
    """grapes_aggregate_rows64_peer_x over each rank's destination window = grapes_aggregate_rows64 over the whole table
    (feature bounds and window bounds differ: the sources of a window are any rows)."""
    from grapes_b200.gcn import ShardedGraphNorm, WideGraphNorm
    from grapes_b200.graph import DeviceGraph
    from grapes_b200.synth import synth_edge_index
    dev = cuda_device
    N = 9000
    gen = torch.Generator().manual_seed(F)
    ei = synth_edge_index(N, 80_000, 5, power_law=1.2)
    g = DeviceGraph.from_edge_index(ei, N, device=dev)
    whole = WideGraphNorm(g)
    x = torch.randn((N, F), generator=gen).to(dev, dtype)
    ldx = (F + 3) // 4 * 4
    bias = torch.randn(F, generator=gen).to(dev)
    for b in (None, bias):
        ref = torch.full((N, F), float("nan"), device=dev)
        whole.aggregate_rows(x, torch.tensor([N, 0], dtype=torch.int32, device=dev), N, ref, bias=b)
        for W in (1, 3, 8):
            tabs, ptrs, bounds = _shards(x, W, ldx)
            out = torch.full((N, F), float("nan"), device=dev)
            for r in range(W):
                p = ShardedGraphNorm(g, W, r)
                for r0 in range(p.lo, p.hi, 1000):
                    n = min(1000, p.hi - r0)
                    slab = torch.tensor([n, r0], dtype=torch.int32, device=dev)
                    p.aggregate_rows_sharded(ptrs, bounds, W, dtype == torch.bfloat16, F, ldx, slab, n, out[r0:], bias=b)
            torch.cuda.synchronize()
            _same(ref, out, f"W {W}")


def _canaries(feats):
    """NaN in every shard's pad columns and behind its last row."""
    for s in feats:
        s.table.rows[:, s.F:] = float("nan")
        s.table.rows[s.hi - s.lo:] = float("nan")


def _engines(dev, W, shape="small", multilabel=False, bf16=False, F=None, **kw):
    from grapes_b200.dist import ShardedFeatures
    from grapes_b200.engine import GrapesEngine
    from grapes_b200.graph import DeviceGraph
    from grapes_b200.synth import SHAPES, make_synth
    cfg = dict(SHAPES[shape])
    d = make_synth(shape, seed=3, multilabel=multilabel, **({"F": F} if F else {}))
    x = d.x.to(dev)
    if bf16:
        x = x.bfloat16()
    g = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=dev)
    feats = ShardedFeatures.emulate(x, W)
    _canaries(feats)
    hp = dict(num_classes=d.num_classes, batch_size=cfg["batch_size"], num_samples=cfg["num_samples"],
              sampling_hops=cfg["sampling_hops"], hidden_dim=256, seed=5)
    hp.update(kw)
    rep = GrapesEngine(g, x, d.y.to(dev), **hp)
    sh = GrapesEngine(g, feats[W - 1], d.y.to(dev), **hp)
    assert sh.ldx == (d.num_features + 3) // 4 * 4 and sh.x is None
    return d, rep, sh


@pytest.mark.parametrize("case", ["tb", "reinforce", "multilabel", "dropout", "bf16", "simt", "wide", "width38"])
def test_step_equals_replicated_engine(cuda_device, case):
    kw = {"tb": {}, "reinforce": dict(reinforce_baseline=True), "multilabel": dict(multilabel=True),
          "dropout": dict(dropout=0.3), "bf16": dict(bf16=True), "simt": dict(use_tensor_cores=False), "wide": {},
          "width38": dict(F=38)}[case]
    d, rep, sh = _engines(cuda_device, 3, **kw)
    if case == "wide":                      # the relabel + build_csr classifier form
        rep.PREP_MAX_ROWS = sh.PREP_MAX_ROWS = 64
        assert rep.cap_A > 64
    t = d.train_mask.nonzero().squeeze(1)[:rep.B].to(torch.int32).to(cuda_device)
    _same(rep.step(t, apply_optim=False, record=True), sh.step(t, apply_optim=False, record=True), case)
    rep.check_overflow(); sh.check_overflow()


def test_graph_replay_prefetch_adam_and_predict(cuda_device):
    """Three optimiser steps through CUDA-graph replays with the next batch prefetched, then predict, W = 8."""
    d, rep, sh = _engines(cuda_device, 8)
    idx = d.train_mask.nonzero().squeeze(1).to(torch.int32).to(cuda_device)
    batches = [b.contiguous() for b in torch.split(idx, rep.B)][:4]
    for eng in (rep, sh):
        for i in range(3):
            eng.step(batches[i], use_graph=True, next_targets=batches[i + 1])
        eng.check_overflow()
    _same(rep.params, sh.params, "params")
    _same(rep.exp_avg, sh.exp_avg, "exp_avg")
    test = d.test_mask.nonzero().squeeze(1).to(torch.int32).to(cuda_device)[:rep.B].contiguous()
    preds = []
    for eng in (rep, sh):
        out = torch.zeros(rep.B, dtype=torch.int32, device=cuda_device)
        eng.predict(test, out)
        eng.check_overflow()
        preds.append(out)
    _same(preds[0], preds[1], "predict")


@pytest.mark.parametrize("name,multilabel,bf16", [("small", False, False), ("small", False, True), ("tiny", True, False),
                                                  ("cora", False, False), ("cora", False, True)])
def test_full_batch_evaluation_equals_one_process(cuda_device, name, multilabel, bf16):
    """W = 2 / 4 / 8 emulated ranks: window logits = the module forward and counts = one-process evaluate(), for F <= D
    (small, tiny) and F > D (cora: P = X W1^T per shard, aggregated from its owners)."""
    from grapes_b200 import eval as E
    from grapes_b200.dist import ShardedFeatures
    from grapes_b200.gcn import (GraphNorm, LocalRowTable, ShardedGraphNorm, _scores_from_counts, needs_p_table,
                                 sharded_layer1, sharded_layer1_p, sharded_layer2)
    from test_gpu_eval_wide import _streamed_setup
    dev = cuda_device
    d, st, g, gcn_c, gcn_gf, args = _streamed_setup(name, 0, dev, multilabel=multilabel)
    gcn_c.eval()
    x = d.x.to(dev)
    if bf16:
        x = x.bfloat16()
        d.x = x
    y = d.y.to(dev)
    mask = (d.val_mask if multilabel else d.test_mask).to(dev)
    ei = d.edge_index.to(dev)
    with torch.no_grad():
        module, _ = gcn_c(x.float(), GraphNorm(g, edge_index=ei))
    want = E.evaluate(gcn_c, gcn_gf, d, args, g, None, st.num_indicators, dev, mask=mask, full_batch=True)
    C, D = d.num_classes, 256
    for W in (2, 4, 8):
        feats = ShardedFeatures.emulate(x, W)
        _canaries(feats)
        assert needs_p_table(gcn_c, feats[0]) == (d.num_features > D)
        parts = [ShardedGraphNorm(g, W, r, edge_index=ei) for r in range(W)]
        ztabs = LocalRowTable.make(W, max(p.rows for p in parts), (C + 3) // 4 * 4, dev)
        ptabs = [None] * W
        if needs_p_table(gcn_c, feats[0]):
            ptabs = LocalRowTable.make(W, max(f.hi - f.lo for f in feats), D, dev)
            for r in range(W):
                sharded_layer1_p(gcn_c, feats[r], ptabs[r], slab_rows=97)
        for p in parts:
            sharded_layer1(gcn_c, feats[p.rank], p, ztabs[p.rank], slab_rows=97, p_table=ptabs[p.rank])
        got, counts = [], torch.zeros(3, dtype=torch.int64, device=dev)
        for p in parts:
            lg, c = sharded_layer2(gcn_c, p, ztabs[p.rank], y=y, mask=mask, return_logits=True)
            got.append(lg)
            counts += c
        _same(torch.cat(got), module, f"W {W}")
        scores = (E._mean_of_hits(int(counts[0]), int(counts[1])),) * 2 if y.dim() == 1 else \
            _scores_from_counts(counts, False)
        assert scores == want, (W, scores, want)


def test_refusals(cuda_device, tmp_path):
    """embed_nodes with a sharded table; full-batch evaluation without a group; a classifier the row-slab forward does not
    cover (no replicated fall-back with a sharded table)."""
    import torch.distributed as dist
    from grapes_b200 import eval as E
    from grapes_b200._lib import GrapesError
    from grapes_b200.dist import ShardedFeatures
    from grapes_b200.engine import GrapesEngine
    from grapes_b200.gcn import GCN
    from test_gpu_eval_wide import _streamed_setup
    dev = cuda_device
    d, st, g, gcn_c, gcn_gf, args = _streamed_setup("tiny", 0, dev)
    feats = ShardedFeatures.emulate(d.x.to(dev), 2)
    with pytest.raises(GrapesError, match="embed_nodes"):
        GrapesEngine(g, feats[0], d.y.to(dev), num_classes=d.num_classes, batch_size=16, num_samples=4,
                     sampling_hops=2, embed_nodes=True)
    with pytest.raises(GrapesError, match="mini-batch"):
        E.evaluate(gcn_c, gcn_gf, d, args, g, None, st.num_indicators, dev, full_batch=True, features=feats[0])
    deep = GCN(d.num_features, [256, 64, d.num_classes]).to(dev).eval()
    narrow = GCN(d.num_features, [4, d.num_classes]).to(dev).eval()       # D <= C
    dist.init_process_group("gloo", init_method=f"file://{tmp_path}/pg", rank=0, world_size=1)
    try:
        for bad in (deep, narrow):
            with pytest.raises(GrapesError, match="mini-batch"):
                E._evaluate_sharded(bad, gcn_gf, d, args, g, st.num_indicators, dev, feats[0], d.y.to(dev),
                                    torch.ones(d.num_nodes, dtype=torch.bool, device=dev), None, True, False, None,
                                    dist.group.WORLD)
    finally:
        dist.destroy_process_group()
