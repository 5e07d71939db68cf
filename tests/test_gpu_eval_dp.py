"""Data-parallel full-batch evaluation on one B200: the per-rank window of the int64 structure (ShardedGraphNorm,
grapes_graph_norm_window_*), the layer-2 aggregation over a row-partitioned operand (grapes_aggregate_rows64_peer) and the
two-phase sharded forward for W emulated ranks, each against the unpartitioned path bit for bit.  The peer kernel does
not care whether its W row bases are peer memory or W allocations of this device, which is what these tests use."""
import pytest
import torch

from test_eval_dp import row_partition
from test_gpu_eval_wide import _hub_edges, _streamed_setup

pytestmark = pytest.mark.gpu


def _graph_case(case):
    from grapes_b200.synth import make_synth, synth_edge_index
    if case in ("tiny", "cora", "small"):
        d = make_synth(case, seed=1)
        return d.num_nodes, d.edge_index
    if case == "multigraph":                  # duplicates, stored self-loops, isolated nodes, hub rows past the sort tiers
        N = 60_000
        ei = torch.cat([synth_edge_index(40_000, 200_000, 3, power_law=1.5), _hub_edges(N, 4)], 1)
        ei[1, :9] = ei[0, :9]
        return N, torch.cat([ei, ei[:, :50_000]], 1)
    return 3, torch.tensor([[0, 1, 2, 2], [1, 2, 0, 2]])            # N < W


@pytest.mark.parametrize("case", ["tiny", "cora", "small", "multigraph", "three_nodes"])
def test_windows_concatenate_to_the_whole_structure(cuda_device, case):
    from grapes_b200.gcn import ShardedGraphNorm, WideGraphNorm
    from grapes_b200.graph import DeviceGraph
    N, ei = _graph_case(case)
    g = DeviceGraph.from_edge_index(ei, N, device=cuda_device)
    for source in ("csr", "edges"):
        kw = {} if source == "csr" else dict(edge_index=ei, chunk_edges=max(ei.shape[1] // 3, 1))
        whole = WideGraphNorm(g, **kw)
        in_off = whole.in_off.cpu()
        weight = (in_off[1:] - in_off[:-1] + 1).numpy()
        for W in (1, 2, 3, 8):
            parts = [ShardedGraphNorm(g, W, r, **kw) for r in range(W)]
            bounds = parts[0].bounds
            assert bounds == row_partition(in_off.numpy(), W)
            assert all(p.bounds == bounds for p in parts)
            assert bounds == ShardedGraphNorm(g, W, W - 1, **kw).bounds        # identical across calls
            for k in range(W):
                assert abs(int(weight[bounds[k]:bounds[k + 1]].sum()) - weight.sum() / W) <= weight.max()
            offs = [p.in_off.cpu() + in_off[p.lo] for p in parts]
            assert torch.equal(torch.cat([o[:-1] for o in offs] + [offs[-1][-1:]]), in_off)
            assert torch.equal(torch.cat([p.in_src.cpu() for p in parts]), whole.in_src.cpu())
            for p in parts:
                assert torch.equal(p.dinv, whole.dinv)
            if N < W:
                assert sum(p.rows == 0 for p in parts) == W - N


def _split(Z, bounds):
    """W separate allocations holding rows bounds[o] .. bounds[o+1] of Z (NaN beyond them: never read)."""
    from grapes_b200.gcn import LocalRowTable
    W = len(bounds) - 1
    rows = max(bounds[o + 1] - bounds[o] for o in range(W))
    tables = LocalRowTable.make(W, rows, Z.shape[1], Z.device)
    for o, t in enumerate(tables):
        t.rows.fill_(float("nan"))
        t.rows[:bounds[o + 1] - bounds[o]] = Z[bounds[o]:bounds[o + 1]]
    return tables


@pytest.mark.parametrize("C", [1, 6, 7, 47, 172])          # 6: the two-float (VEC = 2) form
def test_peer_aggregation_bit_identical_to_rows64(cuda_device, C):
    from grapes_b200._lib import lib
    from grapes_b200.gcn import ShardedGraphNorm, WideGraphNorm
    from grapes_b200.graph import DeviceGraph
    from grapes_b200.synth import synth_edge_index
    dev = cuda_device
    N = 9000
    ei = torch.cat([synth_edge_index(6000, 60_000, 5, power_law=1.0), _hub_edges(N, 2)[:, :8000]], 1)  # 6000.. isolated
    g = DeviceGraph.from_edge_index(ei, N, device=dev)
    whole = WideGraphNorm(g)
    gen = torch.Generator(device=dev).manual_seed(C)
    L = lib()
    for F, ld in ((C, C), ((C + 3) // 4 * 4, (C + 3) // 4 * 4)):
        Z = torch.randn((N, ld), device=dev, generator=gen)
        Z[:, C:] = 0
        for bias in (None, torch.randn(F, device=dev, generator=gen)):
            ref = torch.full((N, F), float("nan"), device=dev)
            whole.aggregate_rows(Z[:, :F] if F != ld else Z, torch.tensor([N, 0], dtype=torch.int32, device=dev), N, ref,
                                 bias=bias)
            L.cdll.grapes_agg_variant(1)
            try:
                ref1 = torch.full((N, F), float("nan"), device=dev)
                whole.aggregate_rows(Z[:, :F] if F != ld else Z, torch.tensor([N, 0], dtype=torch.int32, device=dev), N,
                                     ref1, bias=bias)
            finally:
                L.cdll.grapes_agg_variant(0)
            assert torch.equal(ref, ref1)
            for W in (1, 3, 8):
                parts = [ShardedGraphNorm(g, W, r) for r in range(W)]
                tables = _split(Z, parts[0].bounds)
                out = torch.full((N, F), float("nan"), device=dev)
                for p in parts:
                    for R in (max(p.rows, 1), 777):
                        for r0 in range(p.lo, p.hi, R):
                            n = min(R, p.hi - r0)
                            slab = torch.tensor([n, r0], dtype=torch.int32, device=dev)
                            p.aggregate_rows_peer(tables[p.rank], slab, n, out[r0:], bias=bias)
                assert torch.equal(out, ref), f"F {F} W {W}"
    # zero-row windows: more ranks than rows
    g3 = DeviceGraph.from_edge_index(torch.tensor([[0, 1, 2], [1, 2, 1]]), 3, device=dev)
    w3 = WideGraphNorm(g3)
    Z = torch.randn((3, 4), device=dev, generator=gen)
    ref = torch.empty((3, 4), device=dev)
    w3.aggregate_rows(Z, torch.tensor([3, 0], dtype=torch.int32, device=dev), 3, ref)
    parts = [ShardedGraphNorm(g3, 8, r) for r in range(8)]
    tables = _split(Z, parts[0].bounds)
    out = torch.full((3, 4), float("nan"), device=dev)
    for p in parts:
        slab = torch.tensor([p.rows, p.lo], dtype=torch.int32, device=dev)
        p.aggregate_rows_peer(tables[p.rank], slab, p.rows, out[p.lo:])
    assert torch.equal(out, ref)


@pytest.mark.parametrize("name,seed,multilabel,bf16", [("small", 1, False, False), ("small", 1, False, True),
                                                       ("cora", 0, False, False), ("cora", 0, False, True),
                                                       ("tiny", 3, True, False), ("tiny", 3, True, True)])
def test_emulated_world_equals_one_gpu(cuda_device, name, seed, multilabel, bf16):
    from grapes_b200 import eval as E
    from grapes_b200.gcn import (GraphNorm, LocalRowTable, ShardedGraphNorm, WideGraphNorm, _scores_from_counts,
                                 full_graph_forward_sharded, full_graph_forward_streamed, sharded_layer1, sharded_layer2)
    dev = cuda_device
    d, st, g, gcn_c, gcn_gf, args = _streamed_setup(name, seed, dev, multilabel=multilabel)
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
    streamed, _ = full_graph_forward_streamed(gcn_c, x, WideGraphNorm(g, edge_index=ei))
    assert torch.equal(streamed, module)
    want = E.evaluate(gcn_c, gcn_gf, d, args, g, None, st.num_indicators, dev, mask=mask, full_batch=True)
    C = d.num_classes
    for W in (2, 4, 8):
        parts = [ShardedGraphNorm(g, W, r, edge_index=ei) for r in range(W)]
        rows = max(p.rows for p in parts)
        tables = LocalRowTable.make(W, rows, (C + 3) // 4 * 4, dev)
        for R in (None, 97):
            for p in parts:
                sharded_layer1(gcn_c, x, p, tables[p.rank], slab_rows=R)
            got, counts = [], torch.zeros(3, dtype=torch.int64, device=dev)
            for p in parts:
                lg, c = sharded_layer2(gcn_c, p, tables[p.rank], slab_rows=R, y=y, mask=mask, return_logits=True)
                got.append(lg)
                counts += c
            assert torch.equal(torch.cat(got), module), f"W {W} slab rows {R}"
            scores = (E._mean_of_hits(int(counts[0]), int(counts[1])),) * 2 if y.dim() == 1 else \
                _scores_from_counts(counts, False)
            assert scores == want, (scores, want)
        if W == 2:        # the barrier-separated driver, on a one-rank stand-in table
            solo = ShardedGraphNorm(g, 1, 0, edge_index=ei)
            one = LocalRowTable.make(1, solo.rows, (C + 3) // 4 * 4, dev)[0]
            lg, _ = full_graph_forward_sharded(gcn_c, x, solo, one, return_logits=True)
            assert torch.equal(lg, module)


def test_sharded_forward_refuses_a_table_of_the_wrong_width(cuda_device):
    from grapes_b200._lib import GrapesError
    from grapes_b200.gcn import LocalRowTable, ShardedGraphNorm, sharded_layer1
    d, st, g, gcn_c, gcn_gf, args = _streamed_setup("tiny", 0, cuda_device)
    p = ShardedGraphNorm(g, 2, 0)
    with pytest.raises(GrapesError):
        sharded_layer1(gcn_c.eval(), d.x.to(cuda_device), p, LocalRowTable.make(2, p.rows, 4, cuda_device)[0])
