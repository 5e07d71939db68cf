"""Evaluation parity (SURVEY.md section 8 rows f1, f2): /root/reference/eval.py restated in
oracle/reference_port.py::reference_evaluate vs grapes_b200.eval.evaluate on the device.
Integer outputs (sampled sets, blocks, predictions) bit-exact; logits within 1e-5 of the fp64 oracle."""
import types

import pytest
import torch

from oracle import reference_port as rp

pytestmark = pytest.mark.gpu
TOL = 1e-5


def _close(got, ref, tol=TOL):
    ref = ref.double()
    scale = ref.abs().max().clamp_min(1e-30)
    err = (got.double().cpu() - ref).abs().max() / scale
    assert err < tol, f"relative error {err:.3e} >= {tol}"


def _setup(name, seed, dev, **over):
    from grapes_b200.gcn import GCN
    from grapes_b200.graph import DeviceGraph
    from grapes_b200.synth import make_synth, SHAPES
    cfg = dict(SHAPES[name]); cfg.update(over)
    d = make_synth(name, seed=seed, **over)
    st = rp.OracleState(d, sampling_hops=cfg["sampling_hops"], num_samples=cfg["num_samples"], seed=seed + 7,
                        dtype=torch.float64)
    g = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=dev)
    gcn_c = GCN(d.num_features, [256, d.num_classes]).to(dev)
    gcn_c.load_state_dict({k: v.float() for k, v in st.gcn_c.state_dict().items()})
    gcn_gf = GCN(d.num_features + st.num_indicators, [256, 1]).to(dev)
    gcn_gf.load_state_dict({k: v.float() for k, v in st.gcn_gf.state_dict().items()})
    args = types.SimpleNamespace(sampling_hops=cfg["sampling_hops"], num_samples=cfg["num_samples"], use_indicators=True)
    return cfg, d, st, g, gcn_c, gcn_gf, args


@pytest.mark.parametrize("name,seed", [("tiny", 0), ("cora", 0), ("small", 1)])
def test_full_batch_eval_matches_oracle(cuda_device, name, seed):
    from grapes_b200.eval import evaluate
    cfg, d, st, g, gcn_c, gcn_gf, args = _setup(name, seed, cuda_device)
    ref = rp.reference_evaluate(st, d.test_mask, full_batch=True)
    acc, f1, logits = evaluate(gcn_c, gcn_gf, d, args, g, None, st.num_indicators, cuda_device, mask=d.test_mask,
                               full_batch=True, return_predictions=True)
    _close(logits, ref["logits"])
    pred = torch.argmax(logits, dim=1).cpu()[d.test_mask]
    # argmax may only differ where the oracle's top two logits are closer than the float tolerance
    top2 = ref["logits"][d.test_mask].topk(2, dim=1).values
    safe = (top2[:, 0] - top2[:, 1]) > 1e-4 * ref["logits"].abs().max()
    assert torch.equal(pred[safe], ref["predictions"][safe])
    assert abs(acc - ref["accuracy"]) <= (~safe).sum().item() / max(int(d.test_mask.sum()), 1) + 1e-6
    assert acc == f1


def test_full_batch_eval_multilabel(cuda_device):
    from grapes_b200.eval import evaluate
    cfg, d, st, g, gcn_c, gcn_gf, args = _setup("tiny", 3, cuda_device, multilabel=True)
    ref = rp.reference_evaluate(st, d.val_mask, full_batch=True)
    acc, f1 = evaluate(gcn_c, gcn_gf, d, args, g, None, st.num_indicators, cuda_device, mask=d.val_mask, full_batch=True)
    assert abs(f1 - ref["f1"]) < 1e-6 and acc == f1


def test_graph_norm_matches_edge_list_structure(cuda_device):
    """GraphNorm (whole CSR, TMA-staged kernel at n >= 4096) == NormAdj(edge_index) bit for bit, and both equal the
    register-staged kernel (grapes_agg_variant 1)."""
    from grapes_b200._lib import lib
    from grapes_b200.gcn import GraphNorm, NormAdj
    from grapes_b200.graph import DeviceGraph
    from grapes_b200.synth import make_synth
    d = make_synth("small", seed=2, power_law=1.0)
    ei = d.edge_index.clone()
    ei[:, :7] = ei[0, :7]                                      # stored self-loops: dropped, then one added per node
    g = DeviceGraph.from_edge_index(ei, d.num_nodes, device=cuda_device)
    x = d.x.to(cuda_device)
    gn = GraphNorm(g)
    uniq = torch.unique(ei[0] * d.num_nodes + ei[1])
    ei_u = torch.stack([uniq // d.num_nodes, uniq % d.num_nodes]).to(cuda_device)
    na = NormAdj(ei_u, d.num_nodes)
    assert torch.equal(gn.in_off.cpu()[: d.num_nodes + 1], na.in_off.cpu()[: d.num_nodes + 1])
    assert torch.equal(gn.in_src.cpu(), na.in_src.cpu()[: gn.in_src.numel()])
    assert torch.equal(gn.dinv.cpu(), na.dinv.cpu()[: d.num_nodes])
    L = lib()
    try:
        y_tma = gn.aggregate(x)
        L.cdll.grapes_agg_variant(1)
        y_reg = gn.aggregate(x)
        y_na = na.aggregate(x)
    finally:
        L.cdll.grapes_agg_variant(0)
    assert torch.equal(y_tma, y_reg) and torch.equal(y_tma, y_na)
    _close(y_tma, rp.gcn_conv(d.x.double(), ei_u.cpu(), torch.eye(d.num_features, dtype=torch.float64), None))


@pytest.mark.parametrize("name,seed,bs", [("tiny", 0, 32), ("tiny", 1, 50), ("cora", 0, 512)])
def test_mini_batch_eval_matches_oracle(cuda_device, name, seed, bs):
    from grapes_b200.eval import evaluate
    cfg, d, st, g, gcn_c, gcn_gf, args = _setup(name, seed, cuda_device)
    mask = d.val_mask
    ref = rp.reference_evaluate(st, mask, full_batch=False, batch_size=bs)
    idx = mask.nonzero().squeeze(1)
    loader = [(b,) for b in torch.split(idx, bs)]
    acc, f1, pred = evaluate(gcn_c, gcn_gf, d, args, g, None, st.num_indicators, cuda_device, mask=mask,
                             loader=loader, full_batch=False, return_predictions=True)
    assert torch.equal(pred.cpu(), ref["predictions"])
    assert abs(acc - ref["accuracy"]) < 1e-6 and acc == f1


@pytest.mark.parametrize("name,seed,bs,tc", [("tiny", 0, 32, False), ("small", 1, 128, True), ("small", 2, 100, True)])
def test_mini_batch_eval_engine_path_bit_exact_per_hop(cuda_device, name, seed, bs, tc):
    """The evaluator's batch body on the engine (GrapesEngine.predict, eval.py:84-153): per hop the candidate list, the
    deterministic top-k set and the block in the EVALUATION direction (rows = previous_nodes, cols = targets u sampled,
    eval.py:140-142) bit-exact against the oracle; classifier logits at 1e-5; eager launches == graph replay."""
    from grapes_b200.engine import GrapesEngine
    cfg, d, st, g, gcn_c, gcn_gf, args = _setup(name, seed, cuda_device)
    dev = cuda_device
    mask = d.val_mask
    ref = rp.reference_evaluate(st, mask, full_batch=False, batch_size=bs)
    eng = GrapesEngine(g, d.x.to(dev), d.y.to(dev), num_classes=d.num_classes, batch_size=bs,
                       num_samples=cfg["num_samples"], sampling_hops=cfg["sampling_hops"], use_tensor_cores=tc)
    eng.load_state_dicts(gcn_c=st.gcn_c.state_dict(), gcn_gf=st.gcn_gf.state_dict())
    idx = mask.nonzero().squeeze(1)
    out = torch.zeros(bs, dtype=torch.int32, device=dev)
    out_g = torch.zeros(bs, dtype=torch.int32, device=dev)
    for bi, t in enumerate(torch.split(idx, bs)):
        b = int(t.numel())
        eng.predict(t.to(dev), out, use_graph=False)
        torch.cuda.synchronize()
        eng.check_overflow()
        rb = ref["batches"][bi]
        sizes = eng.hop_sizes()
        for h, (sz, rh) in enumerate(zip(sizes, rb["hops"])):
            hw = eng.hops[h]
            assert torch.equal(hw.nb_nodes[:sz["c"]].cpu().long(), rh["neighbor_nodes"]), f"batch {bi} hop {h}: candidates"
            assert torch.equal(eng.prev[h + 1][b:b + sz["s"]].cpu().long(), rh["sampled"]), f"batch {bi} hop {h}: top-k set"
            blk = torch.stack([hw.blk_src[:sz["blk"]], hw.blk_dst[:sz["blk"]]]).cpu().long()
            assert torch.equal(blk, rh["block_edges"]), f"batch {bi} hop {h}: block (rows = previous_nodes)"
        A = eng.count("A")
        assert torch.equal(eng.all_nodes[:A].cpu().long(), rb["all_nodes"])
        _close(eng.logits_c[:A], rb["logits"])
        eng.predict(t.to(dev), out_g, use_graph=True)
        torch.cuda.synchronize()
        assert torch.equal(out[:b], out_g[:b]), "graph replay differs from eager launches"


def test_train_mini_batch_eval_uses_configured_batch_size(cuda_device):
    """main.py:127-132 builds val_loader / test_loader with args.batch_size -- NOT the size of the last (partial) training
    batch.  After training on a split that is not a multiple of batch_size, the mini-batch evaluation of train() must
    equal the oracle's evaluation of the SAME weights with batch_size = args.batch_size."""
    from grapes_b200.args import Arguments
    from grapes_b200.synth import make_synth
    from grapes_b200 import train as T
    d = make_synth("tiny", seed=5)
    assert int(d.train_mask.sum()) % 32 != 0
    args = Arguments.parse_args(["--dataset", "tiny", "--batch_size", "32", "--num_samples", "8", "--sampling_hops", "2",
                                   "--max_epochs", "1", "--eval_frequency", "5", "--eval_full_batch", "False",
                                   "--eval_on_cpu", "False"])
    f1, *_ = T.train(args, data=d, device=cuda_device)
    eng = T.train.last_engine
    assert eng.bsz != 32 and eng.B == 32                      # the last training batch was partial
    st = rp.OracleState(d, sampling_hops=2, num_samples=8, seed=0, dtype=torch.float64)
    sd = {k: {n: t.detach().cpu().double() for n, t in v.items()} for k, v in eng.state_dicts().items()}
    st.gcn_c.load_state_dict(sd["gcn_c"]); st.gcn_gf.load_state_dict(sd["gcn_gf"])
    ref = rp.reference_evaluate(st, d.test_mask, full_batch=False, batch_size=32)
    assert abs(f1 - ref["f1"]) < 1e-6


@pytest.mark.parametrize("name,seed,over", [("small", 1, {}), ("small", 4, {}),
                                            ("small", 2, dict(multilabel=True)),      # multi-label: 6 sigmoid outputs
                                            ("small", 3, dict(F=37)),                 # F not a multiple of 4: padded pitch
                                            ("cora", 0, dict(N=4100))])               # F = 1433, C = 7; N >= 4096 takes the path
def test_full_graph_forward_tensor_core_path(cuda_device, name, seed, over):
    """gcn.full_graph_forward (GraphNorm built by the library's kernels, hidden layer on grapes_gemm_bias_relu_tc) against
    the float64 oracle at 1e-5 and the structure against the torch-sort builder bit for bit."""
    from grapes_b200.gcn import GraphNorm, full_graph_forward
    cfg, d, st, g, gcn_c, gcn_gf, args = _setup(name, seed, cuda_device, **over)
    gl, gt = GraphNorm(g, builder="lib"), GraphNorm(g, builder="torch")
    N = d.num_nodes
    assert N >= 4096                                           # below that full_graph_forward runs the module forward
    assert torch.equal(gl.in_off[:N + 1], gt.in_off[:N + 1]) and torch.equal(gl.in_src, gt.in_src)
    assert torch.equal(gl.dinv[:N], gt.dinv[:N])
    ge = GraphNorm(g, edge_index=d.edge_index.to(cuda_device), builder="lib")       # duplicates kept, self-loops dropped
    ref = rp.reference_evaluate(st, d.test_mask, full_batch=True)
    logits = full_graph_forward(gcn_c.eval(), d.x.to(cuda_device), ge)
    _close(logits, ref["logits"])


def _builder_case(case):
    """(N, edge_index) of the graph cases of test_gpu_eval_wide.py::test_builder_equals_torch_builder, with stored
    self-loops and duplicated edges"""
    from grapes_b200.synth import make_synth, synth_edge_index
    if case in ("tiny", "cora", "small"):
        N, ei = make_synth(case, seed=1).num_nodes, make_synth(case, seed=1).edge_index
    elif case == "power_law":
        N = 60_000
        gen = torch.Generator().manual_seed(4)
        hubs = [torch.stack([torch.randint(0, N, (d,), generator=gen), torch.full((d,), v, dtype=torch.int64)])
                for v, d in enumerate([40000, 5000, 1500, 600, 100, 50, 20])]     # in-degrees in every sort tier
        ei = torch.cat([synth_edge_index(N, 300_000, 3, power_law=1.5)] + hubs, 1)
    elif case == "isolated":
        N = 9000
        ei = synth_edge_index(4000, 20_000, 5)                    # nodes 4000 .. 8999 have no edge
    else:
        N, ei = 1, torch.zeros((2, 3), dtype=torch.int64)         # one node, three stored self-loops
    ei = ei.clone()
    k = min(7, ei.shape[1])
    ei[1, :k] = ei[0, :k]                                         # stored self-loops: dropped
    return N, torch.cat([ei, ei[:, : ei.shape[1] // 3]], 1)       # duplicates: kept and counted for an edge list


def _lib_or_refusal(graph, **kw):
    """GraphNorm(builder="lib"), or None when it refused with GrapesError because grapes_build_csr flagged overflow bits
    (e.g. more hub rows than the context's worklist): such a build must raise, never return a silent result"""
    from grapes_b200._lib import GrapesError
    from grapes_b200.gcn import GraphNorm
    try:
        return GraphNorm(graph, builder="lib", **kw)
    except GrapesError as e:
        assert "overflow" in str(e), str(e)
        return None


@pytest.mark.parametrize("case", ["tiny", "cora", "small", "power_law", "isolated", "one_node"])
def test_lib_builder_equals_torch_builder(cuda_device, case):
    """GraphNorm(builder="lib") == GraphNorm(builder="torch") bit for bit (in_off, in_src, dinv, nnz), built from the
    graph's CSR (duplicates collapsed) and from the raw edge_index (duplicates kept and counted)"""
    from grapes_b200.gcn import GraphNorm
    from grapes_b200.graph import DeviceGraph
    N, ei = _builder_case(case)
    g = DeviceGraph.from_edge_index(ei, N, device=cuda_device)
    for kw in ({}, dict(edge_index=ei.to(cuda_device))):
        gt = GraphNorm(g, builder="torch", **kw)
        gl = _lib_or_refusal(g, **kw)
        if gl is None:
            continue
        assert gl.n == gt.n == N
        assert int(gl.cnt[0]) == int(gt.cnt[0]) == int(gt.in_src.numel()), "nnz"
        assert torch.equal(gl.in_off[:N + 1], gt.in_off[:N + 1])
        assert torch.equal(gl.in_src[:gt.in_src.numel()], gt.in_src)
        assert torch.equal(gl.dinv[:N], gt.dinv[:N])


def _fp64_forward(gcn, x, indptr, indices):
    """the two-layer GCN forward in float64 on the device over the gcn_norm structure of a canonical CSR (row = source):
    stored self-loops dropped, one self-loop per node added, deg = in-degree + 1"""
    N = x.shape[0]
    src = torch.repeat_interleave(torch.arange(N, device=x.device), indptr[1:] - indptr[:-1])
    dst = indices.long()
    keep = src != dst
    src, dst = src[keep], dst[keep]
    dinv = (torch.bincount(dst, minlength=N) + 1).double().rsqrt()
    loops = torch.arange(N, device=x.device)
    A = torch.sparse_coo_tensor(torch.stack([torch.cat([dst, loops]), torch.cat([src, loops])]),
                                torch.cat([dinv[dst] * dinv[src], dinv * dinv]), (N, N)).coalesce().to_sparse_csr()
    del src, dst, keep
    l0, l1 = gcn.gcn_layers
    h = torch.relu((A @ x.double()) @ l0.lin.weight.double().t() + l0.bias.double())
    return A @ (h @ l1.lin.weight.double().t()) + l1.bias.double()


@pytest.mark.parametrize("name", ["arxiv", "products"])
def test_full_graph_forward_large_synthetic(cuda_device, name):
    """full_graph_forward on the lib-built structure of an ogbn-arxiv- and an ogbn-products-shaped synthetic graph against
    the float64 forward of the same module at 1e-5"""
    from grapes_b200.gcn import GCN, GraphNorm, full_graph_forward
    from grapes_b200.graph import DeviceGraph
    from grapes_b200.synth import make_synth
    dev = cuda_device
    d = make_synth(name, seed=0)
    g = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=dev)
    torch.manual_seed(0)
    gcn = GCN(d.num_features, [256, d.num_classes]).to(dev).eval()
    with torch.no_grad():
        for layer in gcn.gcn_layers:                           # non-zero biases, so both bias adds are checked
            layer.bias.normal_(0.0, 0.1)
    gl = GraphNorm(g, builder="lib")
    x = d.x.to(dev)
    got = full_graph_forward(gcn, x, gl)
    ref = _fp64_forward(gcn, x, g.indptr, g.indices)
    err = ((got.double() - ref).abs().max() / ref.abs().max()).item()
    assert err < TOL, f"relative error {err:.3e}"
