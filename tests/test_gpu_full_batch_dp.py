"""Data-parallel full-graph training on one B200 with emulated ranks: the source windows of the transposed structure
(grapes_graph_norm_t_window_*), the transposed aggregation over a row-partitioned operand, one epoch of W emulated ranks
against float64 with forward logits bit-identical to the module's, the emulated driver against the float64 loop, and
the refusals that come before any allocation.  The peer kernel does not care whether its W row bases are peer memory or
W allocations of this device, which is what these tests use."""
import gc
import types

import pytest
import torch

from directed_utils import directed_synth
from oracle import reference_port as rp
from parity_utils import TOL, _grad_ok, _rel as _rel_cpu
from test_gpu_eval_wide import _hub_edges

pytestmark = pytest.mark.gpu


def _rel(got, ref):
    return _rel_cpu(got.detach().cpu(), ref.detach().cpu())


def _structure_case(case):
    from grapes_b200.synth import synth_edge_index
    if case == "multigraph":        # directed, duplicates, stored self-loops, isolated nodes 40000.., a hub row
        N = 60_000
        ei = torch.cat([synth_edge_index(40_000, 200_000, 3, power_law=1.5)[:, :100_000], _hub_edges(N, 4).flip(0)], 1)
        ei[1, :9] = ei[0, :9]
        return N, torch.cat([ei, ei[:, :30_000]], 1)
    if case == "empty":
        return 500, torch.zeros((2, 0), dtype=torch.int64)
    return 3, torch.tensor([[0, 1, 2, 2, 0], [1, 2, 0, 2, 1]])            # N < W


@pytest.mark.parametrize("case", ["multigraph", "empty", "three_nodes"])
def test_transposed_windows_concatenate_to_the_whole_structure(cuda_device, case):
    from grapes_b200.gcn import ShardedGraphNorm, transposed_structure
    from grapes_b200.graph import DeviceGraph
    N, ei = _structure_case(case)
    E = ei.shape[1]
    g = DeviceGraph.from_edge_index(ei, N, device=cuda_device)
    sources = {"csr": ({}, dict(graph=g)),
               "host": (dict(edge_index=ei, chunk_edges=max(E // 3, 1)), dict(edge_index=ei)),
               "device": (dict(edge_index=ei.to(cuda_device), chunk_edges=max(E // 4, 1)), dict(edge_index=ei))}
    for source, (kw, whole_kw) in sources.items():
        off, dst = transposed_structure(N, cuda_device, **whole_kw)
        off, dst = off.cpu(), dst.cpu()
        for W in (1, 2, 3, 8):
            parts = [ShardedGraphNorm(g, W, r, **kw) for r in range(W)]
            dinv = [p.dinv.clone() for p in parts]
            bounds = [(p.lo, p.hi) for p in parts]
            for p in parts:
                p.build_transposed()
                p.build_transposed()                                   # once
            assert [(p.lo, p.hi) for p in parts] == bounds and parts[0].bounds == ShardedGraphNorm(g, W, 0, **kw).bounds
            offs = [p.out_off.cpu() + off[p.lo] for p in parts]
            assert torch.equal(torch.cat([o[:-1] for o in offs] + [offs[-1][-1:]]), off), (source, W)
            assert torch.equal(torch.cat([p.out_dst.cpu() for p in parts]), dst), (source, W)
            for p, d0 in zip(parts, dinv):
                assert torch.equal(p.dinv, d0)
            if N < W:
                assert sum(p.rows == 0 for p in parts) == W - N


def test_transposed_window_entry_points(cuda_device):
    """The two C entry points called directly: the CSR form over input row ranges split anywhere, the edge form over
    chunks; both equal the rows lo .. hi of the whole transposed structure."""
    from grapes_b200._lib import lib, ptr
    from grapes_b200.gcn import transposed_structure
    from grapes_b200.graph import DeviceGraph
    dev = cuda_device
    N, ei = _structure_case("multigraph")
    g = DeviceGraph.from_edge_index(ei, N, device=dev)
    L, st = lib(), torch.cuda.current_stream(dev).cuda_stream
    for name, lo, hi in (("mid", 17_000, 41_000), ("head", 0, 5), ("one", 59_999, 60_000)):
        for source in ("csr", "edges"):
            ref_off, ref_dst = transposed_structure(N, dev, **(dict(graph=g) if source == "csr" else dict(edge_index=ei)))
            ws = torch.empty(int(L.cdll.grapes_graph_norm_workspace_bytes(N)), dtype=torch.uint8, device=dev)
            err = torch.zeros(1, dtype=torch.int32, device=dev)
            nnz = torch.zeros(1, dtype=torch.int64, device=dev)
            full = torch.empty(N + 1, dtype=torch.int64, device=dev)
            src, dst = ei[0].to(dev).contiguous(), ei[1].to(dev).contiguous()
            L.grapes_graph_norm_begin(N, ptr(ws), ws.numel(), ptr(err), st)
            if source == "csr":
                L.grapes_graph_norm_t_add_csr(0, N, ptr(g.indptr), ptr(g.indices), 0, N, None, None, ptr(ws), ptr(err), st)
            else:
                L.grapes_graph_norm_t_add_edges(0, N, ptr(src), ptr(dst), src.numel(), None, None, ptr(ws), ptr(err), st)
            L.grapes_graph_norm_t_offsets(N, ptr(ws), ptr(full), ptr(nnz), st)
            win = (full[lo:hi + 1] - full[lo]).contiguous()
            out = torch.full((max(int(win[-1]), 1) + 8,), -7, dtype=torch.int32, device=dev)        # canary past the end
            if source == "csr":
                cut = min(lo + 3, N)                                             # one cut inside the window
                for a, b in ((0, cut), (cut, N)):
                    L.grapes_graph_norm_t_window_add_csr(N, ptr(g.indptr), ptr(g.indices), a, b, lo, hi,
                                                         ptr(win), ptr(out), ptr(ws), st)
            else:
                for a in range(0, src.numel(), 70_001):
                    s, d = src[a:a + 70_001], dst[a:a + 70_001]
                    L.grapes_graph_norm_t_window_add_edges(N, ptr(s), ptr(d), s.numel(), lo, hi, ptr(win), ptr(out),
                                                           ptr(ws), st)
                L.grapes_graph_norm_finish(hi - lo, ptr(win), ptr(out), ptr(ws), st)
            assert int(err.item()) == 0
            n = int(win[-1])
            assert torch.equal(win.cpu(), (ref_off[lo:hi + 1] - ref_off[lo]).cpu()), (name, source)
            assert torch.equal(out[:n].cpu(), ref_dst[int(ref_off[lo]):int(ref_off[hi])].cpu()), (name, source)
            assert bool((out[n:] == -7).all()), (name, source)


@pytest.mark.parametrize("C", [1, 7, 47])
def test_peer_transposed_aggregation_bit_identical(cuda_device, C):
    """Rows of A_hat^T G read from the owners of G's rows equal WideGraphNorm.aggregate(G, transpose=True) bit for bit;
    NaN behind every window's rows and in the pad columns is never read; the output's pad columns are zero."""
    from grapes_b200.gcn import LocalRowTable, ShardedGraphNorm, WideGraphNorm
    from grapes_b200.graph import DeviceGraph
    dev = cuda_device
    N, ei = _structure_case("multigraph")
    g = DeviceGraph.from_edge_index(ei, N, device=dev)
    G = torch.randn((N, C), device=dev, generator=torch.Generator(device=dev).manual_seed(C))
    C4 = (C + 3) // 4 * 4
    for kw in ({}, dict(edge_index=ei)):
        ref = WideGraphNorm(g, **kw).aggregate(G, transpose=True)
        for W in (1, 3, 8):
            parts = [ShardedGraphNorm(g, W, r, **kw) for r in range(W)]
            rows = max(p.rows for p in parts)
            tables = LocalRowTable.make(W, rows + 5, C4, dev)
            for p, t in zip(parts, tables):
                t.rows.fill_(float("nan"))
                t.rows[:p.rows, :C] = G[p.lo:p.hi]
            out = torch.full((N, C4), float("nan"), device=dev)
            for p in parts:
                for R in (max(p.rows, 1), 999):
                    for r0 in range(p.lo, p.hi, R):
                        n = min(R, p.hi - r0)
                        slab = torch.tensor([n, r0], dtype=torch.int32, device=dev)
                        p.aggregate_rows_peer(tables[p.rank], slab, n, out[r0:], transpose=True, F=C)
            assert torch.equal(out[:, :C], ref), f"W {W}"
            assert bool((out[:, C:] == 0).all())


# --------------------------------------------------------------------------------------------------------- one epoch
def _epoch_case(case, dev):
    from grapes_b200.synth import make_synth
    if case == "directed_reg":
        return directed_synth("small", 2), 64, 1e-3, False
    if case == "multilabel":
        return make_synth("small", seed=3, multilabel=True), 64, 0., False
    if case == "cora":                                                 # F = 1433 > D
        return make_synth("cora", seed=4), 64, 0., False
    if case == "bf16":
        return directed_synth("small", 5), 64, 1e-3, True
    return make_synth("products", seed=0, device=dev), 256, 0., False


def _oracle_epoch(d, gcn, x, reg, dev):
    """float64 forward + loss + backward of the same classifier on the whole graph (sparse A_hat)"""
    from grapes_b200.full_batch import classifier_loss
    ei, w = rp.gcn_norm(d.edge_index.to(dev), d.num_nodes, dtype=torch.float64)
    A = torch.sparse_coo_tensor(torch.stack([ei[1], ei[0]]), w, (d.num_nodes, d.num_nodes)).coalesce()
    params = {n: p.detach().double().clone().requires_grad_(True) for n, p in gcn.named_parameters()}
    x64 = x.double()
    pre = torch.sparse.mm(A, x64 @ params["gcn_layers.0.lin.weight"].t()) + params["gcn_layers.0.bias"]
    logits = torch.sparse.mm(A, torch.relu(pre) @ params["gcn_layers.1.lin.weight"].t()) + params["gcn_layers.1.bias"]
    loss = classifier_loss(logits, d.y.to(dev), d.train_mask.to(dev), reg)
    loss.backward()
    return logits.detach(), loss.detach(), {n: p.grad for n, p in params.items()}, pre.detach()


def _emulated_epoch(gcn, x, d, W, reg, dev):
    from grapes_b200.full_batch import WindowEpoch, run_epoch_emulated
    from grapes_b200.gcn import LocalRowTable, ShardedGraphNorm
    from grapes_b200.graph import DeviceGraph
    g = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=dev)
    sgns = [ShardedGraphNorm(g, W, r, edge_index=d.edge_index) for r in range(W)]
    rows = max(s.rows for s in sgns)
    D, C = gcn.gcn_layers[0].out_channels, gcn.gcn_layers[1].out_channels
    zt = LocalRowTable.make(W, rows, (C + 3) // 4 * 4, dev)
    dt = LocalRowTable.make(W, rows, D, dev) if x.shape[1] > D else [None] * W
    y, mask = d.y.to(dev), d.train_mask.to(dev)
    epochs = [WindowEpoch(gcn, x, s, z, y, mask, int(mask.sum()), reg, t) for s, z, t in zip(sgns, zt, dt)]
    flat = run_epoch_emulated(epochs)
    logits = torch.cat([e.logits for e in epochs])
    return flat, logits, g


@pytest.mark.parametrize("W", [1, 2, 3, 8])
@pytest.mark.parametrize("case", ["directed_reg", "multilabel", "cora", "bf16"])
def test_epoch_against_float64(cuda_device, case, W):
    _check_epoch(cuda_device, case, W)


def test_products_shaped_epoch_w8(cuda_device):
    _check_epoch(cuda_device, "products", 8)


def _check_epoch(dev, case, W):
    from grapes_b200.full_batch import _set_grads
    from grapes_b200.gcn import GCN, GraphNorm
    d, D, reg, bf16 = _epoch_case(case, dev)
    torch.manual_seed(11)
    gcn = GCN(d.num_features, [D, d.num_classes]).to(dev)
    x = d.x.to(dev)
    if bf16:
        x = x.bfloat16()
    flat, logits, g = _emulated_epoch(gcn, x, d, W, reg, dev)
    with torch.no_grad():
        gn = GraphNorm(g, edge_index=d.edge_index)
        module, _ = gcn(x.float(), gn)
        pre32 = gcn.gcn_layers[0](x.float(), gn)
    assert torch.equal(logits, module), "window logits differ from gcn(x, GraphNorm)"
    loss = _set_grads(gcn, flat)
    r_logits, r_loss, r_grads, pre64 = _oracle_epoch(d, gcn, x.float(), reg, dev)
    assert _rel(logits, r_logits) < TOL
    assert abs(loss.item() - r_loss.item()) < TOL * abs(r_loss.item()), (loss.item(), r_loss.item())
    differ = (pre32 > 0) != (pre64 > 0)                  # relu kinks excuse the layer-1 rows of that unit
    units = set()
    if differ.any():
        assert pre64[differ].abs().max() < 1e-5 * pre64.abs().max(), "relu branch differs from float64 away from a kink"
        units = set(differ.nonzero(as_tuple=True)[1].tolist())
    for n, p in gcn.named_parameters():
        flips = units if n.startswith("gcn_layers.0") else ()
        assert _grad_ok(p.grad, r_grads[n].cpu(), r_grads[n].cpu(), flips), f"gradient {n}"


# ------------------------------------------------------------------------------------------------------------ driver
def _args(**kw):
    from grapes_b200.args import Arguments
    a = Arguments(dataset="synth", hidden_dim=32, max_epochs=3, eval_frequency=2, seed=3, lr_gc=1e-2, runs=1)
    for k, v in kw.items():
        setattr(a, k, v)
    return a


@pytest.mark.parametrize("W", [2, 8])
@pytest.mark.parametrize("case", ["single", "multilabel"])
def test_emulated_driver_against_float64(cuda_device, case, W):
    """The trained parameters against test_gpu_full_graph's float64 loop, under that file's bar."""
    from test_gpu_full_graph import _float64_loop
    from grapes_b200 import full_batch as fb
    from grapes_b200.eval import evaluate
    from grapes_b200.graph import DeviceGraph
    from grapes_b200.synth import make_synth
    if case == "single":
        d, args = directed_synth("small", 5), _args(reg_param=1e-3)
    else:
        d, args = make_synth("small", seed=6, multilabel=True), _args()
    og, _ = _float64_loop(d, args, cuda_device)
    og32, _ = _float64_loop(d, args, cuda_device, torch.float32)
    test_f1, m1, m2, m3 = fb.train_emulated(args, d, cuda_device, W)
    assert len(m1) == len(m2) == len(m3) == args.max_epochs
    got = dict(fb.train.last_model.named_parameters())
    ref32 = dict(og32.named_parameters())
    for n, p in og.named_parameters():
        assert _rel(got[n], p) < max(1e-4, 2 * _rel(ref32[n], p)), n
    g = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=cuda_device)
    _, f1 = evaluate(fb.train.last_model, None, d, args, g, None, 0, cuda_device, mask=d.test_mask, eval_on_cpu=False,
                     full_batch=True)
    assert f1 == test_f1


def test_emulated_driver_is_deterministic_and_frees_its_structure(cuda_device):
    from grapes_b200 import full_batch as fb
    from grapes_b200.synth import make_synth
    runs = []
    for _ in range(2):
        d = make_synth("cora", seed=9)                   # F > D: the d pre table and the P product
        gc.collect()
        before = torch.cuda.memory_allocated(cuda_device)
        gc.disable()
        try:
            f1 = fb.train_emulated(_args(hidden_dim=16), d, cuda_device, 3)[0]
            model = fb.train.last_model
            held = sum(-(-4 * t.numel() // 512) * 512 for p in model.parameters() for t in (p, p.grad))
            assert torch.cuda.memory_allocated(cuda_device) - before <= held, "train_emulated() left memory allocated"
        finally:
            gc.enable()
        runs.append((f1, {n: p.detach().clone() for n, p in model.named_parameters()}))
    assert runs[0][0] == runs[1][0]
    for n in runs[0][1]:
        assert torch.equal(runs[0][1][n], runs[1][1][n]), n


def _meta_papers():
    from grapes_b200.synth import SHAPES
    s = SHAPES["papers"]
    return types.SimpleNamespace(num_nodes=s["N"], num_features=s["F"], num_classes=s["C"],
                                 x=torch.empty((s["N"], s["F"]), dtype=torch.bfloat16, device="meta"),
                                 edge_index=torch.empty((2, s["E_dir"]), dtype=torch.int64, device="meta"))


@pytest.mark.parametrize("why", ["embed_nodes", "dropout", "sharded", "narrow", "working_set"])
def test_refusals_before_any_allocation(cuda_device, why):
    from grapes_b200 import full_batch as fb
    from grapes_b200._lib import GrapesError
    from grapes_b200.dist import ShardedFeatures
    from grapes_b200.synth import make_synth
    d, args, W = make_synth("small", seed=1), _args(), 2
    if why == "embed_nodes":
        args.embed_nodes, match = True, "embed_nodes"
    elif why == "dropout":
        args.dropout, match = 0.5, "dropout"
    elif why == "sharded":
        d.x, match = ShardedFeatures.emulate(d.x, 2, cuda_device)[0], "sharded"
    elif why == "narrow":
        args.hidden_dim, match = d.num_classes - 1, "hidden width"
    else:
        d, args, W, match = _meta_papers(), _args(hidden_dim=256), 1, "bytes"
    gc.collect()
    torch.cuda.synchronize(cuda_device)
    torch.cuda.reset_peak_memory_stats(cuda_device)
    before = torch.cuda.memory_allocated(cuda_device)
    with pytest.raises(GrapesError, match=match):
        fb.train_emulated(args, d, cuda_device, W)
    assert torch.cuda.max_memory_allocated(cuda_device) <= before
