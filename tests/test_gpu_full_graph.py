"""Whole-graph training through the drop-in module: the transposed gcn_norm structure (grapes_graph_norm_t_*), the
transposed aggregation on GraphNorm and WideGraphNorm, GCN autograd on raw edge lists past the small context, one
products-shaped epoch, and the full-graph training driver (grapes_b200.full_batch) against float64."""
import gc

import pytest
import torch
import torch.nn.functional as F

from directed_utils import directed_synth
from oracle import reference_port as rp
from parity_utils import TOL, _rel as _rel_cpu

pytestmark = pytest.mark.gpu


def _rel(got, ref):
    return _rel_cpu(got.detach().cpu(), ref.detach().cpu())


def _graph_norms(d, dev):
    from grapes_b200.gcn import GraphNorm, WideGraphNorm
    from grapes_b200.graph import DeviceGraph
    g = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=dev)
    return g, GraphNorm(g, edge_index=d.edge_index), WideGraphNorm(g, edge_index=d.edge_index)


def _transposed_ref(edge_index, N):
    """torch-sort reference keyed by (source, destination): offsets and destinations, self-loops dropped"""
    src, dst = edge_index[0].long().cpu(), edge_index[1].long().cpu()
    keep = src != dst
    key = torch.sort(src[keep] * N + dst[keep]).values
    off = torch.zeros(N + 1, dtype=torch.int64)
    off[1:] = torch.cumsum(torch.bincount(key // N, minlength=N), 0)
    return off, (key % N).to(torch.int32)


def _graphs():
    from grapes_b200.synth import make_synth
    iso = make_synth("small", seed=3)
    iso.edge_index = iso.edge_index[:, (iso.edge_index < 4000).all(0)]      # nodes 4000.. are isolated
    empty = make_synth("tiny", seed=1)
    empty.edge_index = empty.edge_index[:, :0]
    return {"directed": directed_synth("small", 0), "directed_hub": directed_synth("small", 1, power_law=2.0),
            "undirected": make_synth("small", seed=2), "isolated": iso, "empty": empty}


@pytest.mark.parametrize("name", ["directed", "directed_hub", "undirected", "isolated", "empty"])
def test_transposed_structure_bitwise(cuda_device, name):
    """From an edge list (in chunks smaller than E, host and device) and from the canonical CSR: bit for bit against the
    torch-sort reference; dinv stays the forward's (in-degree + 1)."""
    from grapes_b200.gcn import WideGraphNorm, transposed_structure
    from grapes_b200.graph import DeviceGraph
    d = _graphs()[name]
    N, E = d.num_nodes, d.edge_index.shape[1]
    ref_off, ref_dst = _transposed_ref(d.edge_index, N)
    gn = WideGraphNorm(None, edge_index=d.edge_index, num_nodes=N, device=cuda_device)
    dinv0 = gn.dinv.clone()
    for ei in (d.edge_index, d.edge_index.to(cuda_device)):
        off, dst = transposed_structure(N, cuda_device, edge_index=ei, chunk_edges=max(E // 3 + 1, 1))
        assert torch.equal(off.cpu(), ref_off) and torch.equal(dst.cpu(), ref_dst)
    gn.build_transposed()
    assert torch.equal(gn.out_off.cpu(), ref_off) and torch.equal(gn.out_dst.cpu(), ref_dst)
    assert torch.equal(gn.dinv, dinv0)
    indeg = torch.bincount(d.edge_index[1][d.edge_index[0] != d.edge_index[1]], minlength=N)
    assert torch.equal(dinv0.cpu(), 1.0 / torch.sqrt((indeg + 1).float()))
    # the canonical CSR (duplicates collapsed, scipy's form)
    g = DeviceGraph.from_edge_index(d.edge_index, N, device=cuda_device)
    off, dst = transposed_structure(N, cuda_device, graph=g)
    csr_ei = torch.stack([torch.repeat_interleave(torch.arange(N), (g.indptr[1:] - g.indptr[:-1]).cpu()),
                          g.indices.cpu().long()])
    ref_off, ref_dst = _transposed_ref(csr_ei, N)
    assert torch.equal(off.cpu(), ref_off) and torch.equal(dst.cpu(), ref_dst)


def _dense_adj64(edge_index, N, dev):
    ei, w = rp.gcn_norm(edge_index.to(dev), N, dtype=torch.float64)
    return torch.sparse_coo_tensor(torch.stack([ei[1], ei[0]]), w, (N, N)).coalesce()      # out[dst] += w x[src]


@pytest.mark.parametrize("name", ["directed", "directed_hub", "isolated"])
@pytest.mark.parametrize("width", [7, 32])
def test_transposed_aggregation_float64(cuda_device, name, width):
    d = _graphs()[name]
    N = d.num_nodes
    _, gn, wgn = _graph_norms(d, cuda_device)
    G = torch.randn(N, width, generator=torch.Generator().manual_seed(width)).to(cuda_device)
    A = _dense_adj64(d.edge_index, N, cuda_device)
    ref = torch.sparse.mm(A.t(), G.double())
    a = gn.aggregate(G, transpose=True)
    b = wgn.aggregate(G, transpose=True)
    assert _rel(a, ref) < TOL
    assert torch.equal(a, b), "GraphNorm and WideGraphNorm transposed aggregations differ"
    assert torch.equal(a, gn.aggregate(G, transpose=True)) and torch.equal(b, wgn.aggregate(G, transpose=True))
    assert _rel(wgn.aggregate(G), torch.sparse.mm(A, G.double())) < TOL


def _run_module(gcn, x, adj, y, mask):
    """logits, loss and every gradient (parameters and x) of one forward + backward"""
    gcn.zero_grad()
    xg = x.clone().requires_grad_(True)
    logits, _ = gcn(xg, adj)
    loss = F.cross_entropy(logits[mask], y[mask])
    loss.backward()
    grads = {n: p.grad.clone() for n, p in gcn.named_parameters()}
    grads["x"] = xg.grad.clone()
    return logits.detach(), loss.detach(), grads


def _oracle(d, gcn, x, y, mask, dev, sparse=False):
    """float64 forward + backward of the same module: OracleGCN (index_add gcn_conv) or, for graphs whose [E, hidden]
    gather does not fit, the same arithmetic with a sparse A_hat."""
    og = rp.OracleGCN(x.shape[1], [gcn.gcn_layers[0].out_channels, gcn.gcn_layers[1].out_channels]).double().to(dev)
    og.load_state_dict({k: v.double() for k, v in gcn.state_dict().items()})
    x64 = x.double().clone().requires_grad_(True)
    ei = d.edge_index.to(dev)
    if sparse:
        A = _dense_adj64(d.edge_index, d.num_nodes, dev)
        l1, l2 = og.gcn_layers
        pre = torch.sparse.mm(A, x64 @ l1.lin.weight.t()) + l1.bias
        logits = torch.sparse.mm(A, torch.relu(pre) @ l2.lin.weight.t()) + l2.bias
    else:
        pre = rp.gcn_conv(x64, ei, og.gcn_layers[0].lin.weight, og.gcn_layers[0].bias)
        logits, _ = og(x64, ei)
    loss = F.cross_entropy(logits[mask], y[mask])
    loss.backward()
    grads = {n: p.grad for n, p in og.named_parameters()}
    grads["x"] = x64.grad
    return logits.detach(), loss.detach(), grads, pre.detach()


def _check_against_oracle(d, gcn, x, y, mask, got, dev, sparse=False):
    from parity_utils import _grad_ok
    logits, loss, grads = got
    r_logits, r_loss, r_grads, pre64 = _oracle(d, gcn, x, y, mask, dev, sparse)
    assert _rel(logits, r_logits) < TOL, "logits"
    assert abs(loss.item() - r_loss.item()) < TOL * abs(r_loss.item()), "loss"
    # relu kinks: every hidden (node, unit) whose branch differs from float64 must be a true kink; they excuse the rows of
    # W1 / b1 of that unit and the x-gradient rows of the node's in-neighbours (A_hat^T reaches them)
    with torch.no_grad():
        pre32 = gcn.gcn_layers[0](x, d.edge_index.to(dev))
    differ = (pre32 > 0) != (pre64 > 0)
    units, rows = set(), set()
    if differ.any():
        assert pre64[differ].abs().max() < 1e-5 * pre64.abs().max(), "relu branch differs from float64 away from a kink"
        nodes, u = differ.nonzero(as_tuple=True)
        units = set(u.tolist())
        ei = d.edge_index.to(dev)
        hit = torch.isin(ei[1], nodes)
        rows = set(nodes.tolist()) | set(ei[0][hit].tolist())
    for n, g in grads.items():
        flips = units if n.startswith("gcn_layers.0") else (rows if n == "x" else ())
        assert _grad_ok(g, r_grads[n].cpu(), r_grads[n].cpu(), flips), f"gradient {n}"


@pytest.mark.parametrize("directed", [True, False])
def test_module_autograd_past_the_small_context(cuda_device, directed):
    """GCN(F, [256, C]) on an arxiv-shaped graph (2.3 M edges, past the 2^20 of the small context) with a raw edge_index:
    logits, loss, every parameter gradient and the input gradient against float64; a prebuilt GraphNorm and a
    WideGraphNorm give the same bits as the raw edge list."""
    from grapes_b200.gcn import GCN
    from grapes_b200.synth import make_synth
    from grapes_b200.synth import synth_edge_index
    d = directed_synth("arxiv", 0) if directed else make_synth("arxiv", seed=0)
    if directed:                                                 # one direction of more random pairs: past 2^20 edges
        extra = synth_edge_index(d.num_nodes, d.edge_index.shape[1], seed=11)
        d.edge_index = torch.cat([d.edge_index, extra[:, :extra.shape[1] // 2]], dim=1)
    assert d.edge_index.shape[1] > (1 << 20)
    torch.manual_seed(5)
    gcn = GCN(d.num_features, [256, d.num_classes]).to(cuda_device)
    x, y, mask = d.x.to(cuda_device), d.y.to(cuda_device), d.train_mask.to(cuda_device)
    got = _run_module(gcn, x, d.edge_index.to(cuda_device), y, mask)
    _check_against_oracle(d, gcn, x, y, mask, got, cuda_device)
    _, gn, wgn = _graph_norms(d, cuda_device)
    for adj in (gn, wgn, d.edge_index):                         # prebuilt structures, and a host edge list
        other = _run_module(gcn, x, adj, y, mask)
        assert torch.equal(other[0], got[0]) and torch.equal(other[1], got[1])
        for n in got[2]:
            assert torch.equal(other[2][n], got[2][n]), f"{type(adj).__name__}: gradient {n}"


def test_small_graph_both_paths_bitwise(cuda_device):
    """Inside the small context the raw edge list keeps the NormAdj path; the whole-graph structures give the same logits
    and gradients bit for bit (same arrays, same kernels)."""
    from grapes_b200.gcn import GCN, WideGraphNorm
    d = directed_synth("small", 4)
    torch.manual_seed(6)
    gcn = GCN(d.num_features, [64, d.num_classes]).to(cuda_device)
    x, y, mask = d.x.to(cuda_device), d.y.to(cuda_device), d.train_mask.to(cuda_device)
    ei = d.edge_index.to(cuda_device)
    ref = _run_module(gcn, x, ei, y, mask)
    _, gn, _ = _graph_norms(d, cuda_device)
    wgn = WideGraphNorm(None, edge_index=ei, num_nodes=d.num_nodes, device=cuda_device)
    for adj in (gn, wgn):
        got = _run_module(gcn, x, adj, y, mask)
        assert torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])
        for n in ref[2]:
            assert torch.equal(got[2][n], ref[2][n]), f"{type(adj).__name__}: gradient {n}"
    _check_against_oracle(d, gcn, x, y, mask, ref, cuda_device)


def test_products_shaped_epoch(cuda_device):
    """One whole-graph forward + backward at N = 2.4 M (the split-K weight gradients and the bias column sums over N
    rows), loss and gradients against float64."""
    from grapes_b200.gcn import GCN
    from grapes_b200.synth import make_synth
    d = make_synth("products", seed=0, device=cuda_device)
    torch.manual_seed(7)
    gcn = GCN(d.num_features, [256, d.num_classes]).to(cuda_device)
    got = _run_module(gcn, d.x, d.edge_index, d.y, d.train_mask)
    _check_against_oracle(d, gcn, d.x, d.y, d.train_mask, got, cuda_device, sparse=True)


# ----------------------------------------------------------------------------------------------------------- driver
def _args(**kw):
    from grapes_b200.args import Arguments
    a = Arguments(dataset="synth", hidden_dim=32, max_epochs=3, eval_frequency=2, seed=3, lr_gc=1e-2, runs=1)
    for k, v in kw.items():
        setattr(a, k, v)
    return a


def _float64_loop(d, args, dev, dtype=torch.float64):
    """the driver's epochs restated in float64 (or ``dtype``) from the same initial weights (and table)"""
    from grapes_b200 import full_batch as fb
    F_in = args.node_emb_dim if args.embed_nodes else d.num_features
    init = fb.initial_model(args, F_in, d.num_classes)
    og = rp.OracleGCN(F_in, [args.hidden_dim, d.num_classes]).to(dtype).to(dev)
    og.load_state_dict({k: v.to(dtype) for k, v in init.state_dict().items()})
    params = list(og.parameters())
    if args.embed_nodes:
        x = torch.nn.Parameter(fb.initial_table(args, d.num_nodes).to(dtype).to(dev))
        params.append(x)
    else:
        x = d.x.to(dtype).to(dev)
    opt = torch.optim.Adam(params, lr=args.lr_gc)
    ei, y, mask = d.edge_index.to(dev), d.y.to(dev), d.train_mask.to(dev)
    for _ in range(args.max_epochs):
        logits, _ = og(x, ei)
        loss = fb.classifier_loss(logits, y, mask, args.reg_param)
        opt.zero_grad()
        loss.backward()
        opt.step()
    return og, x


@pytest.mark.parametrize("case", ["single", "multilabel", "embed"])
def test_driver_against_float64(cuda_device, case):
    from grapes_b200 import full_batch as fb
    from grapes_b200.eval import evaluate
    from grapes_b200.graph import DeviceGraph
    from grapes_b200.synth import make_synth
    if case == "single":
        d, args = directed_synth("small", 5), _args(reg_param=1e-3)
    elif case == "multilabel":
        d, args = make_synth("small", seed=6, multilabel=True), _args()
    else:
        d, args = make_synth("tiny", seed=7), _args(embed_nodes=True, node_emb_dim=16)
    og, x64 = _float64_loop(d, args, cuda_device)
    # the bar: 1e-4 after the Adam steps, or -- where the same loop run in fp32 is already further than that from float64
    # (the reg_param term makes the single-label case so) -- no worse than twice that fp32 loop (parity_utils._grad_tol)
    og32, x32 = _float64_loop(d, args, cuda_device, torch.float32)
    test_f1, m1, m2, m3 = fb.train(args, data=d, device=cuda_device)
    assert len(m1) == len(m2) == len(m3) == args.max_epochs
    got = dict(fb.train.last_model.named_parameters())
    ref32 = dict(og32.named_parameters())
    for n, p in og.named_parameters():
        assert _rel(got[n], p) < max(1e-4, 2 * _rel(ref32[n], p)), n
    if args.embed_nodes:
        assert _rel(fb.train.last_table, x64) < max(1e-4, 2 * _rel(x32, x64))
    g = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=cuda_device)
    _, f1 = evaluate(fb.train.last_model, None, d, args, g, None, 0, cuda_device, mask=d.test_mask, eval_on_cpu=False,
                     full_batch=True)
    assert f1 == test_f1


def test_driver_dropout_is_deterministic(cuda_device):
    from grapes_b200 import full_batch as fb
    from grapes_b200.synth import make_synth
    runs = []
    for _ in range(2):
        d = make_synth("small", seed=8)
        gc.collect()
        before = torch.cuda.memory_allocated(cuda_device)
        gc.disable()                  # what train() leaves allocated without the cyclic collector: its model, nothing else
        try:
            f1 = fb.train(_args(dropout=0.5), data=d, device=cuda_device)[0]
            model = fb.train.last_model
            held = sum(-(-4 * t.numel() // 512) * 512 for p in model.parameters() for t in (p, p.grad))
            assert torch.cuda.memory_allocated(cuda_device) - before <= held, "train() left its graph or structure allocated"
        finally:
            gc.enable()
        runs.append((f1, {n: p.detach().clone() for n, p in model.named_parameters()}))
    assert runs[0][0] == runs[1][0]
    for n in runs[0][1]:
        assert torch.equal(runs[0][1][n], runs[1][1][n]), n
    og, _ = _float64_loop(make_synth("small", seed=8), _args(), cuda_device)
    assert _rel(runs[0][1]["gcn_layers.0.lin.weight"], og.gcn_layers[0].lin.weight.detach()) > 1e-3   # dropout acted


def test_driver_refuses_a_papers_shaped_working_set(cuda_device):
    from grapes_b200 import full_batch as fb
    from grapes_b200._lib import GrapesError
    from grapes_b200.synth import SHAPES
    s = SHAPES["papers"]
    # "allocates nothing" is read from the peak: the current count may still drop while the check runs, when the garbage
    # collector frees objects of earlier tests
    gc.collect()
    torch.cuda.synchronize(cuda_device)
    torch.cuda.reset_peak_memory_stats(cuda_device)
    before = torch.cuda.memory_allocated(cuda_device)
    with pytest.raises(GrapesError, match="bytes"):
        fb.check_fits(s["N"], s["E_dir"], s["F"], 256, s["C"], False, cuda_device)
    assert torch.cuda.max_memory_allocated(cuda_device) <= before
    a = SHAPES["arxiv"]
    assert fb.check_fits(a["N"], a["E_dir"], a["F"], 256, a["C"], False, cuda_device) > 0
