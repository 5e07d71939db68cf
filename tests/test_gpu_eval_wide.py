"""Full-batch evaluation past 2^31 edges: the int64 whole-graph structure (WideGraphNorm, grapes_graph_norm_*), the row-slab
aggregation (grapes_aggregate_rows64) and the streamed two-layer forward (full_graph_forward_streamed), against the int32
path (GraphNorm, grapes_aggregate, gcn_c(x, GraphNorm)) bit for bit where that path runs, and against float64
recomputations on a graph of more than 2^31 stored edges."""
import types

import pytest
import torch

from oracle import reference_port as rp

pytestmark = pytest.mark.gpu
TOL = 1e-5


def _close(got, ref, tol=TOL):
    ref = ref.double()
    scale = ref.abs().max().clamp_min(1e-30)
    err = (got.double().cpu() - ref.cpu()).abs().max() / scale
    assert err < tol, f"relative error {err:.3e} >= {tol}"


def _same_structure(w, g):
    N = g.n
    assert torch.equal(w.in_off.cpu(), g.in_off[:N + 1].cpu().long())
    assert torch.equal(w.in_src.cpu(), g.in_src[:g.E].cpu())
    assert torch.equal(w.dinv.cpu(), g.dinv[:N].cpu())


def _hub_edges(N, seed):
    """edges into nodes 0..6 with in-degrees in every sort tier (HBM > 32768, CTA <= 32768, <= 2048, warp <= 1024,
    registers <= 128 / 64 / 32), with repeated sources"""
    gen = torch.Generator().manual_seed(seed)
    parts = []
    for v, d in enumerate([40000, 5000, 1500, 600, 100, 50, 20]):
        src = torch.randint(0, N, (d,), generator=gen)
        parts.append(torch.stack([src, torch.full((d,), v, dtype=torch.int64)]))
    return torch.cat(parts, 1)


@pytest.mark.parametrize("case", ["tiny", "cora", "small", "power_law", "isolated", "one_node"])
def test_builder_equals_torch_builder(cuda_device, case):
    from grapes_b200.gcn import GraphNorm, WideGraphNorm
    from grapes_b200.graph import DeviceGraph
    from grapes_b200.synth import make_synth, synth_edge_index
    if case in ("tiny", "cora", "small"):
        N, ei = make_synth(case, seed=1).num_nodes, make_synth(case, seed=1).edge_index
    elif case == "power_law":
        N = 60_000
        ei = torch.cat([synth_edge_index(N, 300_000, 3, power_law=1.5), _hub_edges(N, 4)], 1)
    elif case == "isolated":
        N = 9000
        ei = synth_edge_index(4000, 20_000, 5)                    # nodes 4000 .. 8999 have no edge
    else:
        N, ei = 1, torch.zeros((2, 3), dtype=torch.int64)         # one node, three stored self-loops
    ei = ei.clone()
    k = min(7, ei.shape[1])
    ei[1, :k] = ei[0, :k]                                         # stored self-loops: dropped
    ei = torch.cat([ei, ei[:, : ei.shape[1] // 3]], 1)            # duplicates: kept and counted for an edge list
    g = DeviceGraph.from_edge_index(ei, N, device=cuda_device)
    _same_structure(WideGraphNorm(g), GraphNorm(g, builder="torch"))
    ref = GraphNorm(g, edge_index=ei.to(cuda_device), builder="torch")
    _same_structure(WideGraphNorm(g, edge_index=ei.to(cuda_device)), ref)
    _same_structure(WideGraphNorm(g, edge_index=ei, chunk_edges=max(ei.shape[1] // 5, 1)), ref)   # host, in chunks


def test_builder_rejects_ids_outside_the_graph(cuda_device):
    from grapes_b200._lib import GrapesError
    from grapes_b200.gcn import WideGraphNorm
    from grapes_b200.graph import DeviceGraph
    ei = torch.tensor([[0, 1, 2], [1, 2, 0]])
    g = DeviceGraph.from_edge_index(ei, 3, device=cuda_device)
    with pytest.raises(GrapesError, match="outside"):
        WideGraphNorm(g, edge_index=torch.tensor([[0, 1, 5], [1, 2, 0]]))


def _agg_cases():
    for F in (100, 128, 602, 1433):
        for bf16 in (False, True):
            for bias in (False, True):
                yield F, bf16, bias


@pytest.mark.parametrize("F,bf16,bias", list(_agg_cases()))
def test_rows64_bit_identical_to_int32_aggregation(cuda_device, F, bf16, bias):
    """grapes_aggregate_rows64 over r0 = 0 and r0 > 0 slabs == grapes_aggregate(_bf16) on the int32 structure, in the
    TMA-staged form (variant 0) and the register-staged one (variant 1), with a contiguous and a padded row pitch."""
    from grapes_b200._lib import lib, ptr
    from grapes_b200.gcn import GraphNorm, WideGraphNorm
    from grapes_b200.graph import DeviceGraph
    from grapes_b200.synth import make_synth
    from grapes_b200.utils import _stream
    dev = cuda_device
    d = make_synth("small", seed=2, power_law=1.0, features=False)
    N = d.num_nodes
    g = DeviceGraph.from_edge_index(d.edge_index, N, device=dev)
    gn, wn = GraphNorm(g, builder="torch"), WideGraphNorm(g)
    gen = torch.Generator(device=dev).manual_seed(F)
    b = torch.randn(F, device=dev, generator=gen) if bias else None
    L = lib()
    pitches = [F, (F + 7) // 8 * 8 + 8]
    try:
        for variant in (0, 1):
            L.cdll.grapes_agg_variant(variant)
            for ldx in pitches:
                store = torch.randn((N, ldx), device=dev, generator=gen)
                if bf16:
                    store = store.bfloat16()
                x = store[:, :F]
                ref = torch.empty((N, F), dtype=torch.float32, device=dev)
                fn = L.grapes_aggregate_bf16 if bf16 else L.grapes_aggregate
                fn(g.ctx, ptr(x), F, ldx, None, gn.cnt.data_ptr() + 4, N, ptr(gn.in_off), ptr(gn.in_src), ptr(gn.dinv),
                   None, 0, ptr(b), 0, ptr(ref), F, None, None, -1, _stream())
                for R in (N, 4096, 1000, 333):
                    out = torch.full((N, F), float("nan"), device=dev)
                    for r0 in range(0, N, R):
                        n = min(R, N - r0)
                        slab = torch.tensor([n, r0], dtype=torch.int32, device=dev)
                        wn.aggregate_rows(x, slab, n, out[r0:], bias=b)
                    assert torch.equal(out, ref), f"variant {variant} ldx {ldx} slab {R}"
    finally:
        L.cdll.grapes_agg_variant(0)


def _streamed_setup(name, seed, dev, multilabel=False):
    from grapes_b200.gcn import GCN
    from grapes_b200.graph import DeviceGraph
    from grapes_b200.synth import make_synth, SHAPES
    cfg = dict(SHAPES[name])
    d = make_synth(name, seed=seed, multilabel=multilabel)
    st = rp.OracleState(d, sampling_hops=cfg["sampling_hops"], num_samples=cfg["num_samples"], seed=seed + 7,
                        dtype=torch.float64)
    g = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=dev)
    gcn_c = GCN(d.num_features, [256, d.num_classes]).to(dev)
    gcn_c.load_state_dict({k: v.float() for k, v in st.gcn_c.state_dict().items()})
    gcn_gf = GCN(d.num_features + st.num_indicators, [256, 1]).to(dev)
    gcn_gf.load_state_dict({k: v.float() for k, v in st.gcn_gf.state_dict().items()})
    args = types.SimpleNamespace(sampling_hops=cfg["sampling_hops"], num_samples=cfg["num_samples"], use_indicators=True)
    return d, st, g, gcn_c, gcn_gf, args


@pytest.mark.parametrize("name,seed", [("tiny", 0), ("cora", 0), ("small", 1)])
def test_streamed_forward_bit_identical_to_current_path(cuda_device, name, seed):
    from grapes_b200.gcn import GraphNorm, WideGraphNorm, full_graph_forward_streamed
    d, st, g, gcn_c, gcn_gf, args = _streamed_setup(name, seed, cuda_device)
    ei = d.edge_index.to(cuda_device)
    x = d.x.to(cuda_device)
    gcn_c.eval()
    with torch.no_grad():
        ref, _ = gcn_c(x, GraphNorm(g, edge_index=ei))
    wn = WideGraphNorm(g, edge_index=ei)
    N = d.num_nodes
    y, mask = d.y.to(cuda_device), d.test_mask.to(cuda_device)
    want = (torch.argmax(ref[mask], 1) == y[mask]).float().mean().item()
    for R in (N, 7, 1000, None):
        logits, (acc, f1) = full_graph_forward_streamed(gcn_c, x, wn, slab_rows=R, y=y, mask=mask)
        assert torch.equal(logits, ref), f"slab rows {R}"
        assert acc == want and f1 == acc
        none, scores = full_graph_forward_streamed(gcn_c, x, wn, slab_rows=R, y=y, mask=mask, return_logits=False)
        assert none is None and scores == (acc, f1)


@pytest.mark.parametrize("name,seed,multilabel", [("tiny", 0, False), ("cora", 0, False), ("small", 1, False),
                                                  ("tiny", 3, True)])
def test_evaluate_wide_path_equals_current_path(cuda_device, monkeypatch, name, seed, multilabel):
    from grapes_b200 import eval as E
    d, st, g, gcn_c, gcn_gf, args = _streamed_setup(name, seed, cuda_device, multilabel=multilabel)
    mask = d.val_mask if multilabel else d.test_mask
    cur = E.evaluate(gcn_c, gcn_gf, d, args, g, None, st.num_indicators, cuda_device, mask=mask, full_batch=True,
                     return_predictions=True)
    monkeypatch.setattr(E, "WIDE_MIN_EDGES", 0)
    wide = E.evaluate(gcn_c, gcn_gf, d, args, g, None, st.num_indicators, cuda_device, mask=mask, full_batch=True,
                      return_predictions=True)
    assert type(g._graph_norm[1]).__name__ == "WideGraphNorm"
    assert wide[:2] == cur[:2] and torch.equal(wide[2], cur[2])
    assert E.evaluate(gcn_c, gcn_gf, d, args, g, None, st.num_indicators, cuda_device, mask=mask,
                      full_batch=True) == cur[:2]
    ref = rp.reference_evaluate(st, mask, full_batch=True)
    _close(wide[2], ref["logits"])
    if multilabel:
        assert abs(wide[1] - ref["f1"]) < 1e-6


def test_streamed_forward_refuses_what_it_does_not_cover(cuda_device):
    from grapes_b200._lib import GrapesError
    from grapes_b200.gcn import GCN, WideGraphNorm, full_graph_forward_streamed
    d, st, g, gcn_c, gcn_gf, args = _streamed_setup("tiny", 0, cuda_device)
    wn = WideGraphNorm(g)
    x = d.x.to(cuda_device)
    with pytest.raises(GrapesError):
        full_graph_forward_streamed(GCN(d.num_features, [64, 64, d.num_classes]).to(cuda_device), x, wn)
    with pytest.raises(GrapesError):
        full_graph_forward_streamed(GCN(d.num_features, [256, d.num_classes], dropout=0.5).to(cuda_device).train(), x, wn)


def test_train_reaches_the_same_test_f1_on_the_wide_path(cuda_device, monkeypatch):
    from grapes_b200 import eval as E
    from grapes_b200 import train as T
    from grapes_b200.args import Arguments
    from grapes_b200.synth import make_synth
    argv = ["--dataset", "small", "--batch_size", "128", "--num_samples", "32", "--sampling_hops", "2", "--max_epochs", "2",
            "--eval_frequency", "1", "--eval_full_batch", "True", "--eval_on_cpu", "False"]
    f1_cur, *_ = T.train(Arguments.parse_args(argv), data=make_synth("small", seed=6), device=cuda_device)
    monkeypatch.setattr(E, "WIDE_MIN_EDGES", 0)
    f1_wide, *_ = T.train(Arguments.parse_args(argv), data=make_synth("small", seed=6), device=cuda_device)
    assert f1_wide == f1_cur


S_STRIDE = 479_001


def _strided_csr(N, deg, dev, chunk=1 << 22):
    """row i -> (i + j S) mod N, j = 1 .. deg (S odd, N a power of two: distinct, no self-loop).  Every node has in-degree
    deg and in(v) = {(v - j S) mod N}: the transpose in closed form."""
    indices = torch.empty(N * deg, dtype=torch.int32, device=dev)
    j = torch.arange(1, deg + 1, device=dev, dtype=torch.int64) * S_STRIDE
    for r0 in range(0, N, chunk):
        i = torch.arange(r0, min(N, r0 + chunk), device=dev, dtype=torch.int64)
        indices[r0 * deg:(r0 + i.numel()) * deg] = ((i.unsqueeze(1) + j) % N).reshape(-1).to(torch.int32)
    indptr = torch.arange(N + 1, device=dev, dtype=torch.int64) * deg
    return indptr, indices


def _in_list(v, N, deg):
    return torch.sort((v - torch.arange(1, deg + 1, dtype=torch.int64) * S_STRIDE) % N).values


def _checksum(rows, cols):
    r, c = rows.long(), cols.long()
    return int((r * 1_000_003 + c * 7919 + r * c).sum())


def test_past_2_31_structure_aggregation_and_evaluate(cuda_device):
    """2^25 nodes x 65 = 2.18e9 stored edges, a bf16 table of 128 features: the builder (closed form, checksum, memory
    bound), the row-slab aggregation at rows whose offsets lie past 2^31 (float64 at 1e-5), and evaluate(full_batch=True)
    unforced: logits of sampled mask rows against a float64 recomputation over their two-hop receptive field, the accuracy
    against their argmax, and a peak below table + structure + Z + slab (no fp32 copy of the table)."""
    from grapes_b200._lib import lib
    from grapes_b200.eval import evaluate
    from grapes_b200.gcn import GCN, WideGraphNorm, slab_rows_for
    dev = cuda_device
    N, deg, F, C, D = 1 << 25, 65, 128, 19, 256
    indptr, indices = _strided_csr(N, deg, dev)
    nnz = N * deg
    assert nnz > (1 << 31)
    g = types.SimpleNamespace(indptr=indptr, indices=indices, num_nodes=N, nnz=nnz, device=dev)

    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    wn = WideGraphNorm(g)
    torch.cuda.synchronize()
    ws = int(lib().cdll.grapes_graph_norm_workspace_bytes(N))
    outputs = 8 * (N + 1) + 4 * nnz + 4 * N
    assert torch.cuda.max_memory_allocated() - base <= outputs + ws + (8 << 20)
    assert wn.E == nnz
    assert torch.equal(wn.in_off, torch.arange(N + 1, device=dev, dtype=torch.int64) * deg)
    assert torch.equal(wn.dinv, 1.0 / torch.sqrt(torch.full((N,), float(deg + 1), device=dev)))
    first_high = (1 << 31) // deg + 1
    gen = torch.Generator().manual_seed(0)
    sample = torch.unique(torch.cat([torch.tensor([0, N - 1, first_high - 1, first_high]),
                                     torch.randint(0, N, (24,), generator=gen),
                                     torch.randint(first_high, N - 4096, (24,), generator=gen)]))
    for v in sample.tolist():
        assert torch.equal(wn.in_src[v * deg:(v + 1) * deg].cpu().long(), _in_list(v, N, deg)), f"row {v}"
    fwd = tcs = 0
    for r0 in range(0, N, 1 << 22):
        r1 = min(N, r0 + (1 << 22))
        rows = torch.arange(r0, r1, device=dev).repeat_interleave(deg)
        fwd += _checksum(rows, indices[r0 * deg:r1 * deg])               # (src, dst) of the forward CSR
        tcs += _checksum(wn.in_src[r0 * deg:r1 * deg], rows)            # (src, dst) of the transpose
    assert fwd == tcs

    x = (torch.randn((N, F), generator=torch.Generator().manual_seed(1)) * 0.5).bfloat16().to(dev)
    xd = lambda ids: x[ids.to(dev)].double().cpu()                      # noqa: E731  the bf16-rounded features
    w = 1.0 / (deg + 1)
    # row-slab aggregation at rows past 2^31 entries
    high = sample[sample >= first_high]
    r0 = int(high[0])
    out = torch.empty((4096, F), device=dev)
    wn.aggregate_rows(x, torch.tensor([4096, r0], dtype=torch.int32, device=dev), 4096, out)
    for v in range(r0, r0 + 4096, 511):
        ids = torch.cat([torch.tensor([v]), _in_list(v, N, deg)])
        _close(out[v - r0], xd(ids).sum(0) * w)

    gcn_c = GCN(F, [D, C]).to(dev).eval()
    y = torch.randint(0, C, (N,), device=dev)
    mask = torch.zeros(N, dtype=torch.bool, device=dev)
    mask[sample.to(dev)] = True
    data = types.SimpleNamespace(x=x, y=y, num_nodes=N)
    args = types.SimpleNamespace(sampling_hops=2, num_samples=16, use_indicators=True)
    W1, b1 = gcn_c.gcn_layers[0].lin.weight.double().cpu(), gcn_c.gcn_layers[0].bias.double().cpu()
    W2, b2 = gcn_c.gcn_layers[1].lin.weight.double().cpu(), gcn_c.gcn_layers[1].bias.double().cpu()

    def ref_logits(v):
        us = torch.cat([torch.tensor([v]), _in_list(v, N, deg)])
        hs = []
        for u in us.tolist():
            ts = torch.cat([torch.tensor([u]), _in_list(u, N, deg)])
            hs.append(torch.relu((xd(ts).sum(0) * w) @ W1.T + b1) @ W2.T)
        return torch.stack(hs).sum(0) * w + b2

    ref = torch.stack([ref_logits(v) for v in sample.tolist()])
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()                                 # table + graph + y + mask + model
    torch.cuda.reset_peak_memory_stats()
    acc, f1 = evaluate(gcn_c, None, data, args, g, None, 0, dev, mask=mask.cpu(), full_batch=True)
    C4 = (C + 3) // 4 * 4
    R = slab_rows_for(N, 4 * (F + D + C4), 0, dev, mem_budget=1 << 62)
    bound = outputs + ws + N * C4 * 4 + R * 4 * (F + D + C4) + (64 << 20)
    assert torch.cuda.max_memory_allocated() - base < bound                  # an fp32 copy of the table alone is 4 N F
    acc2, f12, logits = evaluate(gcn_c, None, data, args, g, None, 0, dev, mask=mask.cpu(), full_batch=True,
                                 return_predictions=True)
    assert (acc2, f12) == (acc, f1) and acc == f1
    got = logits[sample.to(dev)].double().cpu()
    _close(got, ref)
    top2 = ref.topk(2, dim=1).values
    safe = (top2[:, 0] - top2[:, 1]) > 1e-4 * ref.abs().max()
    ys = y[sample.to(dev)].cpu()
    assert torch.equal(got.argmax(1)[safe], ref.argmax(1)[safe])
    # the mask is the sampled rows: the accuracy is the argmax hit rate over them (rows too close to call may go either way)
    hits_ref = (ref.argmax(1) == ys)
    lo = (hits_ref & safe).sum().item() / len(sample)
    hi = (hits_ref | ~safe).sum().item() / len(sample)
    assert lo - 1e-6 <= acc <= hi + 1e-6
    assert abs(acc - (got.argmax(1) == ys).double().mean().item()) < 1e-6
