"""Whole training step and evaluation on DIRECTED graphs against the float64 oracle.

Every other parity test runs on make_synth's graphs, which hold both directions of every pair: such a graph is its own
transpose, so a swapped source and destination, or an out-degree used for an in-degree, gives the same numbers there.
The reference builds its CSR from edge_index as given (main.py:134-136) and keeps most datasets directed.  A directed
graph also has rows that are expanded (previous_nodes) and frontier nodes at once while having no out-edge -- a node
that another row points to -- which a symmetric graph never has.  The transposed scalar aggregation of the sampler's
backward must still write their dz; the buffers are filled with a large finite sentinel before the step so that a row
left unwritten shows up in the first step (NaN would not do: rows past the count are legitimately multiplied by 0).

Seeds are chosen so that the fp32 and fp64 oracles select the same sets with a well separated top-k boundary."""
import pytest
import torch

from directed_utils import directed_synth, empty_expanded_frontier_rows
from oracle import reference_port as rp
from parity_utils import TOL, _rel, check_step

pytestmark = pytest.mark.gpu

SENTINEL = 1e3


def _setup(name, seed, dev, use_tensor_cores=False, power_law=0.0, **hp_over):
    from grapes_b200.engine import GrapesEngine
    from grapes_b200.graph import DeviceGraph
    from grapes_b200.synth import SHAPES
    cfg = SHAPES[name]
    torch.manual_seed(1000 + seed)            # the oracle draws its Gumbel noise from the global CPU generator
    d = directed_synth(name, seed, power_law)
    hp = dict(sampling_hops=cfg["sampling_hops"], num_samples=cfg["num_samples"])
    hp.update(hp_over)
    st = rp.OracleState(d, seed=seed + 100, dtype=torch.float64, **hp)
    st.fp32 = rp.OracleState(d, seed=seed + 100, dtype=torch.float32, **hp)
    g = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=dev)
    eng = GrapesEngine(g, d.x.to(dev), d.y.to(dev), num_classes=d.num_classes, batch_size=cfg["batch_size"],
                       hidden_dim=256, lr_gc=1e-3, lr_gf=1e-4, seed=seed, use_tensor_cores=use_tensor_cores, **hp)
    eng.load_state_dicts(gcn_c=st.gcn_c.state_dict(), gcn_gf=st.gcn_gf.state_dict(), gcn_z=st.gcn_z.state_dict())
    _poison_dz(eng)
    train_idx = d.train_mask.nonzero().squeeze(1)
    return d, st, eng, train_idx, cfg["batch_size"]


def _poison_dz(eng):
    for state in eng._states:
        for hw in state["hops"]:
            hw.dz.fill_(SENTINEL)
    if getattr(eng, "dz_z", None) is not None:
        eng.dz_z.fill_(SENTINEL)


def _dz_ref(e_src, e_dst, dinv, dl):
    """float64 A_hat^T dl on the hop graph: dz[j] = dinv[j]^2 dl[j] + sum_{j -> d, d != j} dinv[j] dinv[d] dl[d]"""
    s, t = e_src.cpu().long(), e_dst.cpu().long()
    keep = s != t
    s, t = s[keep], t[keep]
    dinv, dl = dinv.cpu().double(), dl.cpu().double()
    return (dinv * dinv * dl).index_add(0, s, dinv[s] * dinv[t] * dl[t])


def _check_dz_in_every_recorded_step(eng):
    """Holds each recorded step's dz (every hop) and dz_z (gcn_z, trajectory balance) to float64 A_hat^T dl on the
    engine's own hop graph, right after the step and before check_step compares the gradients those vectors feed:
    an unwritten row is then reported as dz rather than as a gradient."""
    step = eng.step

    def checked(*args, **kw):
        rec = step(*args, **kw)
        if rec is not None:
            for h, r in enumerate(rec["hops"]):
                assert _rel(r["dz"], _dz_ref(r["e_src"], r["e_dst"], r["dinv"], r["dl_all"])) < TOL, \
                    f"hop {h}: dz of the sampler backward differs from float64 A_hat^T dl"
            if not (eng.reinforce or eng.random_sampling):
                r = rec["hops"][0]
                n = r["n"]
                dl = torch.full((n,), 1.0 / n, dtype=torch.float64)
                assert _rel(eng.dz_z[:n], _dz_ref(r["e_src"], r["e_dst"], r["dinv"], dl)) < TOL, \
                    "gcn_z: dz_z differs from float64 A_hat^T (1/n)"
        return rec

    eng.step = checked


def _assert_case_present(st, ref):
    for h, b in enumerate(ref["hops"]):
        assert empty_expanded_frontier_rows(st.adjacency, b["prev"], b["batch_nodes"]) > 0, \
            f"hop {h} has no expanded frontier row without out-edges: the graph does not test that case"


@pytest.mark.parametrize("name,seed,tc,reinforce", [
    ("tiny", 0, False, False), ("small", 1, False, False), ("cora", 0, False, False),
    ("tiny", 0, True, False), ("small", 1, True, False), ("cora", 0, True, False),
    ("tiny", 3, False, True), ("small", 1, True, True),
])
def test_directed_step_parity(cuda_device, name, seed, tc, reinforce):
    d, st, eng, train_idx, B = _setup(name, seed, cuda_device, use_tensor_cores=tc, reinforce_baseline=reinforce)
    _check_dz_in_every_recorded_step(eng)
    rec, ref = check_step(st, eng, train_idx[:B], cuda_device, apply_optim=False)
    _assert_case_present(st, ref)


@pytest.mark.parametrize("tc", [False, True])
def test_directed_step_parity_power_law(cuda_device, tc):
    """Zipf-like endpoints: hub rows with thousands of out-edges next to rows with none."""
    d, st, eng, train_idx, B = _setup("small", 6, cuda_device, use_tensor_cores=tc, power_law=1.5)
    _check_dz_in_every_recorded_step(eng)
    rec, ref = check_step(st, eng, train_idx[:B], cuda_device, apply_optim=False)
    _assert_case_present(st, ref)


def test_directed_two_steps_with_adam(cuda_device):
    """Two optimiser steps (test_gpu_engine.py::test_three_steps_with_adam's bars): the second step runs on buffers
    the first one left behind, so a row unwritten there would carry the first step's value."""
    d, st, eng, train_idx, B = _setup("cora", 2, cuda_device)
    _check_dz_in_every_recorded_step(eng)
    nsteps = 2
    for i in range(nsteps):
        check_step(st, eng, train_idx[i * B:(i + 1) * B], cuda_device, apply_optim=True, post_optim=(i > 0))
    for key, net, net32, lr in (("gcn_c", st.gcn_c, st.fp32.gcn_c, 1e-3), ("gcn_gf", st.gcn_gf, st.fp32.gcn_gf, 1e-4),
                                ("gcn_z", st.gcn_z, st.fp32.gcn_z, 1e-4)):
        for (name, p), (_, p32) in zip(net.named_parameters(), net32.named_parameters()):
            ref = p.detach().double()
            got = eng.state_dicts()[key][name].double().cpu()
            err = (got - ref).abs()
            assert err.max() <= 2.0 * lr * nsteps * 1.01, f"{key} {name}: beyond the Adam sign-flip bound"
            scale = ref.abs().max().clamp_min(1e-30)
            frac = (err > 1e-4 * scale).double().mean().item()
            frac32 = ((p32.detach().double() - ref).abs() > 1e-4 * scale).double().mean().item()
            assert frac <= max(0.01, 3.0 * frac32), f"{key} {name}: {frac:.4f} of the weights off by > 1e-4"


def test_directed_graph_replay_matches_eager(cuda_device):
    d, st, eng, train_idx, B = _setup("cora", 0, cuda_device)
    d2, st2, eng2, _, _ = _setup("cora", 0, cuda_device)
    for i in range(2):
        t = train_idx[i * B:(i + 1) * B].to(cuda_device)
        eng.step(t, use_graph=False)
        eng2.step(t, use_graph=True)
        torch.cuda.synchronize()
        assert torch.equal(eng.scal, eng2.scal), f"step {i}: losses differ between eager and graph replay"
    eng.check_overflow(); eng2.check_overflow()
    for name in ("rng_state", "grads", "params", "exp_avg", "exp_avg_sq"):
        assert torch.equal(getattr(eng, name), getattr(eng2, name)), name


def _eval_setup(name, seed, dev):
    from grapes_b200.gcn import GCN
    from grapes_b200.graph import DeviceGraph
    from grapes_b200.synth import SHAPES
    cfg = SHAPES[name]
    d = directed_synth(name, seed)
    st = rp.OracleState(d, sampling_hops=cfg["sampling_hops"], num_samples=cfg["num_samples"], seed=seed + 7,
                        dtype=torch.float64)
    g = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=dev)
    gcn_c = GCN(d.num_features, [256, d.num_classes]).to(dev)
    gcn_c.load_state_dict({k: v.float() for k, v in st.gcn_c.state_dict().items()})
    return cfg, d, st, g, gcn_c


@pytest.mark.parametrize("name,seed,bs,tc", [("tiny", 0, 32, False), ("small", 1, 128, True)])
def test_directed_mini_batch_eval_engine_path_bit_exact_per_hop(cuda_device, name, seed, bs, tc):
    """GrapesEngine.predict (eval.py:84-153): candidates, deterministic top-k set and the block in the evaluation
    direction (rows = previous_nodes) bit-exact per hop; classifier logits at 1e-5; eager == graph replay."""
    from grapes_b200.engine import GrapesEngine
    cfg, d, st, g, gcn_c = _eval_setup(name, seed, cuda_device)
    dev = cuda_device
    mask = d.val_mask
    ref = rp.reference_evaluate(st, mask, full_batch=False, batch_size=bs)
    eng = GrapesEngine(g, d.x.to(dev), d.y.to(dev), num_classes=d.num_classes, batch_size=bs,
                       num_samples=cfg["num_samples"], sampling_hops=cfg["sampling_hops"], use_tensor_cores=tc)
    eng.load_state_dicts(gcn_c=st.gcn_c.state_dict(), gcn_gf=st.gcn_gf.state_dict())
    out = torch.zeros(bs, dtype=torch.int32, device=dev)
    out_g = torch.zeros(bs, dtype=torch.int32, device=dev)
    for bi, t in enumerate(torch.split(mask.nonzero().squeeze(1), bs)):
        b = int(t.numel())
        eng.predict(t.to(dev), out, use_graph=False)
        torch.cuda.synchronize()
        eng.check_overflow()
        rb = ref["batches"][bi]
        for h, (sz, rh) in enumerate(zip(eng.hop_sizes(), rb["hops"])):
            hw = eng.hops[h]
            assert torch.equal(hw.nb_nodes[:sz["c"]].cpu().long(), rh["neighbor_nodes"]), f"batch {bi} hop {h}: candidates"
            assert torch.equal(eng.prev[h + 1][b:b + sz["s"]].cpu().long(), rh["sampled"]), f"batch {bi} hop {h}: top-k set"
            blk = torch.stack([hw.blk_src[:sz["blk"]], hw.blk_dst[:sz["blk"]]]).cpu().long()
            assert torch.equal(blk, rh["block_edges"]), f"batch {bi} hop {h}: block (rows = previous_nodes)"
        A = eng.count("A")
        assert torch.equal(eng.all_nodes[:A].cpu().long(), rb["all_nodes"])
        assert _rel(eng.logits_c[:A], rb["logits"]) < TOL
        eng.predict(t.to(dev), out_g, use_graph=True)
        torch.cuda.synchronize()
        assert torch.equal(out[:b], out_g[:b]), "graph replay differs from eager launches"


@pytest.mark.parametrize("name,seed", [("tiny", 0), ("cora", 0), ("small", 1)])
def test_directed_full_batch_eval(cuda_device, name, seed):
    """eval.py:50 on a graph that differs from its transpose: messages flow from source to destination, degrees are
    in-degrees over edge_index with its duplicates counted."""
    from grapes_b200.eval import evaluate
    import types
    cfg, d, st, g, gcn_c = _eval_setup(name, seed, cuda_device)
    args = types.SimpleNamespace(sampling_hops=cfg["sampling_hops"], num_samples=cfg["num_samples"], use_indicators=True)
    ref = rp.reference_evaluate(st, d.test_mask, full_batch=True)
    acc, f1, logits = evaluate(gcn_c, None, d, args, g, None, st.num_indicators, cuda_device, mask=d.test_mask,
                               full_batch=True, return_predictions=True)
    assert _rel(logits, ref["logits"]) < TOL


def test_directed_graph_norm_matches_edge_list_structure(cuda_device):
    """GraphNorm of the CSR == NormAdj of its (unique) edge list bit for bit on a directed graph, and its aggregation
    equals float64 gcn_conv with identity weights -- in-neighbours are the SOURCES of the edges into a node."""
    from grapes_b200.gcn import GraphNorm, NormAdj
    from grapes_b200.graph import DeviceGraph
    d = directed_synth("small", 2, power_law=1.0)
    N = d.num_nodes
    g = DeviceGraph.from_edge_index(d.edge_index, N, device=cuda_device)
    gn = GraphNorm(g)
    uniq = torch.unique(d.edge_index[0] * N + d.edge_index[1])
    ei_u = torch.stack([uniq // N, uniq % N])
    na = NormAdj(ei_u.to(cuda_device), N)
    assert torch.equal(gn.in_off.cpu()[:N + 1], na.in_off.cpu()[:N + 1])
    assert torch.equal(gn.in_src.cpu(), na.in_src.cpu()[:gn.in_src.numel()])
    assert torch.equal(gn.dinv.cpu(), na.dinv.cpu()[:N])
    x = d.x.to(cuda_device)
    y_gn, y_na = gn.aggregate(x), na.aggregate(x)
    assert torch.equal(y_gn, y_na)
    y_ref = rp.gcn_conv(d.x.double(), ei_u, torch.eye(d.num_features, dtype=torch.float64), None)
    assert _rel(y_gn, y_ref) < TOL
    y_t = rp.gcn_conv(d.x.double(), ei_u.flip(0), torch.eye(d.num_features, dtype=torch.float64), None)
    assert _rel(y_ref, y_t) > 1e-2, "the graph does not differ from its transpose"
