"""CPU tests (no GPU): the oracle against the golden vectors generated from the reference's own code
(tests/golden/make_golden.py), against the reference imported live when GRAPES_REFERENCE_ROOT names a checkout of it,
and against closed forms for the un-vendored PyG GCNConv arithmetic."""
import glob
import os

import numpy as np
import pytest
import torch

from grapes_b200.synth import make_synth
from oracle import ref_import
from oracle import reference_port as rp

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
needs_reference = pytest.mark.skipif(not ref_import.reference_available(),
                                     reason="needs GRAPES_REFERENCE_ROOT: a checkout of the reference GRAPES project")


def _t(a):
    return torch.from_numpy(np.asarray(a))


@pytest.fixture
def single_thread():
    """One CPU thread: scatter-adds / reductions run in a fixed order, so two runs of the same arithmetic agree bit for
    bit and a live-reference comparison can be exact."""
    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    yield
    torch.set_num_threads(threads)


def test_tensormap_docstring_golden():
    """utils.py:104-108 -- the only known-answer vector the reference holds."""
    z = np.load(os.path.join(GOLDEN, "tensormap_docstring.npz"))
    nodes = torch.tensor([22, 32, 42, 52])
    tm = rp.TensorMap(size=nodes.max() + 1)
    tm.update(nodes)
    got = tm.map(_t(z["keys"]))
    assert got.tolist() == z["mapped"].tolist() == [3, 2, 1, 0, 0]


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "hoploop_*.npz"))))
def test_oracle_matches_reference_golden(path):
    z = np.load(path)
    N, k, hops = int(z["N"]), int(z["k"]), int(z["hops"])
    adj = rp.build_adjacency(_t(z["edge_index"]), N)
    assert np.array_equal(adj.indptr, z["csr_indptr"]) and np.array_equal(adj.indices, z["csr_indices"])
    target = _t(z["target_nodes"])
    node_map = rp.TensorMap(N)
    prev = target.clone()
    all_mask = torch.zeros(N, dtype=torch.bool)
    all_mask[target] = True
    for hop in range(hops):
        p = f"hop{hop}_"
        assert torch.equal(prev, _t(z[p + "prev"]))
        nb = rp.get_neighborhoods(prev, adj)
        assert torch.equal(nb, _t(z[p + "neighborhoods"]))
        pm = torch.zeros(N, dtype=torch.bool); bm = torch.zeros(N, dtype=torch.bool)
        pm[prev] = True; bm[nb.view(-1)] = True
        batch_nodes = node_map.values[bm]
        neighbor_nodes = node_map.values[bm & ~pm]
        assert torch.equal(batch_nodes, _t(z[p + "batch_nodes"]))
        assert torch.equal(neighbor_nodes, _t(z[p + "neighbor_nodes"]))
        node_map.update(batch_nodes)
        assert torch.equal(node_map.map(nb), _t(z[p + "local_neighborhoods"]))
        logits = _t(z[p + "logits"])
        noise = _t(z[p + "gumbel"]) if z[p + "gumbel"].size else None
        for stable in (False, True):
            sampled, lp, stats = rp.sample_neighborhoods_from_probs(logits, neighbor_nodes, k, gumbel_noise=noise,
                                                                    stable_ties=stable)
            assert torch.equal(sampled, _t(z[p + "sampled"]))
            assert torch.equal(lp, _t(z[p + "log_prob"]))
            if stats:
                got = [float(stats[s]) for s in ("min_prob", "max_prob", "mean_entropy", "std_entropy")]
                assert np.allclose(got, z[p + "stats"], rtol=0, atol=0)
        all_mask[sampled] = True
        nxt = torch.cat([target, sampled])
        assert torch.equal(rp.slice_adjacency(adj, nxt, prev), _t(z[p + "block_edges"]))
        prev = nxt
    all_nodes = node_map.values[all_mask]
    node_map.update(all_nodes)
    assert torch.equal(all_nodes, _t(z["all_nodes"]))
    assert torch.equal(node_map.map(target), _t(z["local_target_ids"]))


@needs_reference
@pytest.mark.parametrize("name,seed", [("tiny", 3), ("cora", 1), ("small", 0)])
def test_oracle_matches_live_reference(name, seed):
    ru = ref_import.load_reference_utils()
    d = make_synth(name, seed=seed)
    adj_ref = ref_import.reference_adjacency(d.edge_index, d.num_nodes)
    adj = rp.build_adjacency(d.edge_index, d.num_nodes)
    g = torch.Generator().manual_seed(seed)
    for P in (1, 7, 200):
        nodes = torch.randperm(d.num_nodes, generator=g)[:P]
        assert torch.equal(ru.get_neighborhoods(nodes, adj_ref), rp.get_neighborhoods(nodes, adj))
        cols = torch.randperm(d.num_nodes, generator=g)[:P + 3]
        assert torch.equal(ru.slice_adjacency(adj_ref, nodes, cols), rp.slice_adjacency(adj, nodes, cols))
    for n, k in ((500, 16), (40, 64), (2000, 256)):
        logits = torch.randn(n, 1, generator=g)
        nb = torch.arange(n) * 2
        torch.manual_seed(seed)
        a = ru.sample_neighborhoods_from_probs(logits, nb, k)
        torch.manual_seed(seed)
        b = rp.sample_neighborhoods_from_probs(logits, nb, k, stable_ties=False)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and a[2].keys() == b[2].keys()
        for key in a[2]:
            assert torch.equal(a[2][key], b[2][key])


def test_gcn_conv_dense_closed_form():
    """PyG GCNConv == D^-1/2 (A_noloop + I) D^-1/2 X W^T + b with deg = in-degree incl. the loop."""
    g = torch.Generator().manual_seed(0)
    n = 40
    ei = torch.randint(0, n, (2, 150), generator=g)
    ei[:, :4] = ei[0, :4]                                   # explicit self-loops are replaced, not doubled
    ei = torch.cat([ei, ei[:, 10:14]], dim=1)               # duplicate edges are KEPT by PyG
    x = torch.randn(n, 9, dtype=torch.float64, generator=g)
    W = torch.randn(5, 9, dtype=torch.float64, generator=g)
    b = torch.randn(5, dtype=torch.float64, generator=g)
    A = torch.zeros(n, n, dtype=torch.float64)
    for s, t in ei.t().tolist():
        if s != t:
            A[t, s] += 1
    A += torch.eye(n, dtype=torch.float64)
    Dm = torch.diag(A.sum(1).pow(-0.5))
    ref = Dm @ A @ Dm @ x @ W.t() + b
    assert torch.allclose(rp.gcn_conv(x, ei, W, b), ref, atol=1e-12)


def test_gcn_conv_hand_computed_4_nodes():
    """edges 0->1, 0->2, 3->2 (+ a self-loop 1->1 that is dropped).  deg = [1, 2, 3, 1]."""
    ei = torch.tensor([[0, 0, 3, 1], [1, 2, 2, 1]])
    x = torch.tensor([[1.0], [2.0], [3.0], [4.0]], dtype=torch.float64)
    W = torch.tensor([[2.0]], dtype=torch.float64)
    out = rp.gcn_conv(x, ei, W, torch.tensor([0.5], dtype=torch.float64))
    h = 2 * x.squeeze(1)
    want = torch.tensor([h[0] / 1,
                         h[1] / 2 + h[0] / (1 * 2) ** 0.5,
                         h[2] / 3 + h[0] / (1 * 3) ** 0.5 + h[3] / (1 * 3) ** 0.5,
                         h[3] / 1]) + 0.5
    assert torch.allclose(out.squeeze(1), want, atol=1e-12)


def test_reference_step_runs_and_is_deterministic_given_noise():
    d = make_synth("tiny", seed=0)
    tr = d.train_mask.nonzero().squeeze(1)[:32]
    st = rp.OracleState(d, sampling_hops=2, num_samples=8, seed=1)
    rec = rp.reference_step(st, tr, apply_optim=False)
    noise = [h["noise"] for h in rec["hops"]]
    st2 = rp.OracleState(d, sampling_hops=2, num_samples=8, seed=1)
    rec2 = rp.reference_step(st2, tr, gumbel_noise=noise, apply_optim=False)
    assert torch.equal(rec["loss_gfn"], rec2["loss_gfn"])
    for a, b in zip(rec["hops"], rec2["hops"]):
        assert torch.equal(a["sampled"], b["sampled"])
    # trajectory-balance closed form used by the CUDA path: d loss / d logit_i = 2 r (mask_i - p_i)
    r = rec["log_z"] + rec["tot_log_prob"] + st.loss_coef * rec["loss_c"]
    assert torch.allclose(rec["loss_gfn"], r * r, rtol=1e-6)


def test_oracle_embed_nodes_table_is_in_optimizer_c():
    """main.py:89-100,116: the learned table sits in optimizer_c; its gradient after loss_c.backward() is non-zero only on
    all_nodes rows, and torch's dense Adam keeps moving rows of EARLIER batches (what grapes_adam_embed reproduces)."""
    from grapes_b200.synth import make_synth, SHAPES
    cfg = SHAPES["tiny"]
    d = make_synth("tiny", seed=0)
    torch.manual_seed(7)
    st = rp.OracleState(d, sampling_hops=cfg["sampling_hops"], num_samples=cfg["num_samples"], seed=1, embed_nodes=True)
    assert any(p is st.x for g in st.opt_c.param_groups for p in g["params"])
    idx = d.train_mask.nonzero().squeeze(1)
    B = cfg["batch_size"]
    x0 = st.x.detach().clone()
    r1 = rp.reference_step(st, idx[:B])
    outside = torch.ones(d.num_nodes, dtype=torch.bool)
    outside[r1["all_nodes"]] = False
    assert float(r1["grad_x"][outside].abs().max()) == 0.0 and float(r1["grad_x"].abs().max()) > 0.0
    x1 = st.x.detach().clone()
    assert torch.equal(x1[outside], x0[outside]) and not torch.equal(x1, x0)
    r2 = rp.reference_step(st, idx[B:2 * B])
    only_first = torch.zeros(d.num_nodes, dtype=torch.bool)
    only_first[r1["all_nodes"]] = True
    only_first[r2["all_nodes"]] = False
    moved = (st.x.detach()[only_first] != x1[only_first]).any(dim=1)
    assert only_first.any() and bool(moved.any())                  # zero gradient this step, Adam momentum still moves them


def test_csr_oracle_is_the_reference_statement():
    """main.py:134-136 verbatim (``sp.csr_matrix((np.ones(E, dtype=bool), edge_index), shape=(N, N))``) against the
    oracle's ``build_adjacency`` and against a sort/unique restatement in numpy: the three agree on indptr / indices, so
    the GPU tests of grapes_csr_from_edges (tests/test_gpu_csr_build.py) are pinned to what the reference itself builds.
    Row slicing of the reference's (non-canonicalised) matrix gives the same neighbour lists (utils.py:78)."""
    import numpy as np
    import scipy.sparse as sp
    g = torch.Generator().manual_seed(11)
    N, E = 200, 3000
    ei = torch.randint(0, N, (2, E), generator=g)
    ei = torch.cat([ei, ei[:, :500], torch.arange(N).repeat(2, 1)], dim=1)          # duplicates + self-loops
    ref = sp.csr_matrix((np.ones(ei.shape[1], dtype=bool), ei.numpy()), shape=(N, N))   # the reference's statement
    adj = rp.build_adjacency(ei, N)
    key = np.unique(ei[0].numpy() * N + ei[1].numpy())
    rows, cols = key // N, key % N
    indptr = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=N))])
    assert np.array_equal(adj.indptr, indptr) and np.array_equal(adj.indices, cols)
    canon = ref.copy(); canon.sum_duplicates(); canon.sort_indices()
    assert np.array_equal(canon.indptr, adj.indptr) and np.array_equal(canon.indices, adj.indices)
    nodes = torch.tensor([3, 77, 3, 199])
    a = rp.get_neighborhoods(nodes, ref)
    b = rp.get_neighborhoods(nodes, adj)
    assert torch.equal(a, b)


def test_csr_from_edge_index_has_no_cpu_path():
    from grapes_b200._lib import GrapesError
    from grapes_b200.graph import csr_from_edge_index
    with pytest.raises(GrapesError):
        csr_from_edge_index(torch.zeros(2, 3, dtype=torch.long), 4, "cpu")


def test_full_graph_logits_cpu_equals_gcn_conv_path():
    """bench.py's full-graph CPU leg (one sparse-CSR x dense product per layer) is the same arithmetic as the oracle's
    GCN.forward on the deduplicated edge list (eval.py:50)."""
    import numpy as np
    from grapes_b200.synth import make_synth
    d = make_synth("small", seed=1)
    st = rp.OracleState(d, sampling_hops=2, num_samples=8, seed=3, dtype=torch.float64)
    coo = st.adjacency.tocoo()
    ei = torch.stack([torch.from_numpy(coo.row.astype(np.int64)), torch.from_numpy(coo.col.astype(np.int64))])
    with torch.no_grad():
        a = st.gcn_c(st.x, ei)[0]
        b = rp.full_graph_logits_cpu(st.gcn_c, st.x, st.adjacency)
    assert float((a - b).abs().max() / a.abs().max()) < 1e-6


def _eval_state(name, seed, k, hops, weights=None):
    d = make_synth(name, seed=seed)
    st = rp.OracleState(d, sampling_hops=hops, num_samples=k, seed=seed + 5, dtype=torch.float32)
    if weights is not None:
        for key, net in (("gcn_c", st.gcn_c), ("gcn_gf", st.gcn_gf)):
            net.load_state_dict({n: _t(weights[f"w_{key}.{n}"]) for n in net.state_dict()})
    st.gcn_c.eval(); st.gcn_gf.eval()
    return d, st


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "eval_*.npz"))))
def test_oracle_evaluate_matches_reference_golden(path):
    """eval.py:11-165 (SURVEY.md section 8 rows f1 / f2): the fixtures were produced by the reference's OWN ``evaluate``
    (tests/golden/make_golden.py::main_eval); the oracle's restatement must rebuild the same evaluation blocks (bit-exact,
    local ids, evaluation direction), the same logits per batch and the same scores."""
    z = np.load(path)
    name, seed, B, k, hops = str(z["name"]), int(z["seed"]), int(z["B"]), int(z["k"]), int(z["hops"])
    d, st = _eval_state(name, seed, k, hops, weights=z)
    mask = _t(z["mask"])
    assert torch.equal(mask, d.test_mask)
    full = rp.reference_evaluate(st, mask, full_batch=True)
    assert np.allclose(full["logits"].numpy(), z["full_logits"], rtol=0, atol=1e-5 * np.abs(z["full_logits"]).max())
    assert full["accuracy"] == pytest.approx(float(z["full_accuracy"]), abs=1e-12)
    assert full["f1"] == pytest.approx(float(z["full_f1"]), abs=1e-12)
    mini = rp.reference_evaluate(st, mask, full_batch=False, batch_size=B)
    assert len(mini["batches"]) == int(z["mini_batches"])
    for b, rec in enumerate(mini["batches"]):
        node_map = rp.TensorMap(d.num_nodes)
        node_map.update(rec["all_nodes"])
        for h, hop in enumerate(rec["hops"]):
            assert torch.equal(node_map.map(hop["block_edges"]), _t(z[f"mini_b{b}_edges{h}"])), (b, h)
        ref = z[f"mini_b{b}_logits"]
        assert np.allclose(rec["logits"].numpy(), ref, rtol=0, atol=1e-5 * np.abs(ref).max())
    assert mini["accuracy"] == pytest.approx(float(z["mini_accuracy"]), abs=1e-12)
    assert mini["f1"] == pytest.approx(float(z["mini_f1"]), abs=1e-12)


@needs_reference
@pytest.mark.parametrize("name,seed,B,k,hops", [("tiny", 3, 32, 8, 2), ("small", 0, 200, 32, 3), ("cora", 1, 512, 16, 2)])
def test_oracle_evaluate_matches_live_reference_eval(single_thread, name, seed, B, k, hops):
    """The reference's own ``evaluate`` imported live (oracle/ref_import.py::load_reference_eval), full-batch and mini-batch,
    against ``reference_evaluate`` on the same models: scores equal, and every logit the reference's ``gcn_c`` call produced
    equal bit for bit (same CPU arithmetic on the same blocks in the same order)."""
    import argparse
    mod, ru = ref_import.load_reference_eval()
    d, st = _eval_state(name, seed, k, hops)
    args = argparse.Namespace(sampling_hops=hops, use_indicators=True, num_samples=k)
    adj = ref_import.reference_adjacency(d.edge_index, d.num_nodes)
    for mask in (d.test_mask, d.val_mask):
        for full in (True, False):
            loader = torch.utils.data.DataLoader(torch.utils.data.TensorDataset(mask.nonzero().squeeze(1)), batch_size=B)
            rc, rg = ref_import.RecordingModule(st.gcn_c), ref_import.RecordingModule(st.gcn_gf)
            acc, f1 = mod.evaluate(rc, rg, d, args, adj, ru.TensorMap(size=d.num_nodes), hops + 1, torch.device("cpu"),
                                   mask=mask, eval_on_cpu=True, loader=loader, full_batch=full)
            o = rp.reference_evaluate(st, mask, full_batch=full, batch_size=B)
            assert o["accuracy"] == pytest.approx(acc, abs=1e-12) and o["f1"] == pytest.approx(f1, abs=1e-12)
            if full:
                assert torch.equal(rc.calls[0]["logits"], o["logits"])
            else:
                assert len(rc.calls) == len(o["batches"]) and len(rg.calls) == hops * len(rc.calls)
                for c, b in zip(rc.calls, o["batches"]):
                    assert torch.equal(c["logits"], b["logits"])
                    assert torch.equal(c["x"], st.x[b["all_nodes"]])


TRAIN_CASES = {                     # name -> (graph, seed, batch, k, hops, data overrides, argument overrides)
    "tb":        ("tiny", 0, 32, 8, 2, {}, {}),
    "reinforce": ("tiny", 1, 50, 4, 3, {}, {"reinforce_baseline": True}),
    "random":    ("tiny", 2, 32, 8, 2, {}, {"random_sampling": True}),
    "reg_logz":  ("tiny", 3, 40, 6, 2, {}, {"reg_param": 0.1, "log_z_init": 0.7, "loss_coef": 100.0}),
    "multilabel": ("tiny", 4, 32, 8, 2, {"multilabel": True}, {}),
    "small":     ("small", 1, 512, 32, 3, {}, {}),
}


def _oracle_epoch(d, seed, B, k, hops, over, rng_seed, epochs=1):
    """The oracle's batch loop with the global RNG consumed exactly as main.py consumes it: one DataLoader iterator per
    epoch (its base seed is drawn from the global generator, main.py:126,157) and the Gumbel draws of utils.py:40-41."""
    st = rp.OracleState(d, sampling_hops=hops, num_samples=k, seed=seed + 100, dtype=torch.float32, **over)
    torch.manual_seed(rng_seed)
    tr = d.train_mask.nonzero().squeeze(1)
    recs = []
    for _ in range(epochs):
        for batch in torch.utils.data.DataLoader(torch.utils.data.TensorDataset(tr), batch_size=B):
            recs.append(rp.reference_step(st, batch[0], stable_ties=False))
    return st, recs


def _flat_weights(nets):
    return {f"{key}.{n}": p.detach().clone() for key, net in zip(("gcn_c", "gcn_gf", "gcn_z"), nets)
            for n, p in net.named_parameters()}


@needs_reference
@pytest.mark.parametrize("case", sorted(TRAIN_CASES))
def test_oracle_step_matches_live_reference_train(single_thread, case):
    """The reference's OWN ``train(args)`` (main.py:57-340: batch loop, hop loop, both losses, autograd backward, both Adam
    optimisers, final evaluation) executed live from the reference's main.py (oracle/ref_import.py::load_reference_train)
    against the oracle's ``reference_step`` on the same data, initial weights and RNG stream: every batch's loss_c / loss_gfn /
    log_z / sum of log-probs and sampler statistics equal BIT FOR BIT, the weights of all three networks after the epoch equal
    to 1e-7 (autograd accumulates two of them in another order), the test score equal.  Pins SURVEY.md section 8 rows a2-a13
    of the oracle to the reference itself -- except the arithmetic inside GCNConv, which is the oracle's restatement in both
    runs (torch_geometric is absent)."""
    name, seed, B, k, hops, dover, over = TRAIN_CASES[case]
    d = make_synth(name, seed=seed, **dover)
    rng_seed = 4242 + seed
    test_f1, logs, nets = ref_import.run_reference_train(d, weight_seed=seed + 100, rng_seed=rng_seed, batch_size=B,
                                                         num_samples=k, sampling_hops=hops, **over)
    st, recs = _oracle_epoch(d, seed, B, k, hops, over, rng_seed)
    assert len(recs) == len(logs) and len(recs) >= 2
    for r, l in zip(recs, logs):
        assert float(r["loss_c"]) == l["batch_loss_c"]
        assert float(r["loss_gfn"]) == float(l["batch_loss_gfn"])
        assert float(r["log_z"]) == float(l["log_z"].detach())
        assert -float(r["tot_log_prob"]) == float(l["-log_probs"].detach())
        for h, hop in enumerate(r["hops"]):
            for key, v in (hop["stats"] or {}).items():
                assert float(v) == float(l["stats"][f"{key}_{h}"]), (h, key)
    ref_w, got_w = _flat_weights(nets), _flat_weights((st.gcn_c, st.gcn_gf, st.gcn_z))
    for key in ref_w:
        assert torch.allclose(got_w[key], ref_w[key], rtol=0, atol=1e-7 * float(ref_w[key].abs().max())), key
    multilabel = d.y.dim() == 2
    o = rp.reference_evaluate(st, d.test_mask, full_batch=True)
    assert o["f1"] == pytest.approx(test_f1, abs=1e-12) and (multilabel or 0.0 < test_f1 < 1.0)


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "train_*.npz"))))
def test_oracle_step_matches_reference_train_golden(single_thread, path):
    """The fixtures hold what the reference's OWN ``train(args)`` logged and left behind (tests/golden/make_golden.py::
    main_train); the oracle's batch loop must reproduce the losses of every batch, the weights after the epoch and the test
    score from the same seeds (the RNG stream and the initial weights are functions of the seeds)."""
    import json
    z = np.load(path)
    name, seed, B, k, hops = str(z["name"]), int(z["seed"]), int(z["B"]), int(z["k"]), int(z["hops"])
    dover, over = json.loads(str(z["data_overrides"])), json.loads(str(z["arg_overrides"]))
    d = make_synth(name, seed=seed, **dover)
    st, recs = _oracle_epoch(d, seed, B, k, hops, over, 4242 + seed)
    assert len(recs) == len(z["loss_c"])
    for key, ref in (("loss_c", z["loss_c"]), ("loss_gfn", z["loss_gfn"]), ("log_z", z["log_z"])):
        got = np.array([float(r[key]) for r in recs])
        assert np.allclose(got, ref, rtol=1e-6, atol=1e-7), key
    got = np.array([-float(r["tot_log_prob"]) for r in recs])
    assert np.allclose(got, z["neg_log_probs"], rtol=1e-6, atol=1e-7)
    for key, net in (("gcn_c", st.gcn_c), ("gcn_gf", st.gcn_gf), ("gcn_z", st.gcn_z)):
        for n, p in net.named_parameters():
            ref = z[f"w_{key}.{n}"]
            assert np.abs(p.detach().numpy() - ref).max() <= 1e-6 * max(np.abs(ref).max(), 1e-30), (key, n)
    o = rp.reference_evaluate(st, d.test_mask, full_batch=True)
    assert o["f1"] == pytest.approx(float(z["test_f1"]), abs=1e-12)


@needs_reference
def test_oracle_multi_epoch_and_minibatch_eval_match_live_reference_train(single_thread):
    """Four epochs of the reference's own ``train`` with its mid-training validation (main.py:313-326: epoch 4 with
    eval_frequency 5) and the final test evaluation both in MINI-BATCH mode (eval_full_batch=False): the TensorMap and the
    mask buffers are shared between training and evaluation (main.py:102,138-140), the loaders' base seeds come from the
    global RNG.  Losses of all 16 batches bit-equal, final score equal to the oracle's mini-batch ``reference_evaluate``."""
    name, seed, B, k, hops = "tiny", 6, 32, 8, 2
    d = make_synth(name, seed=seed)
    test_f1, logs, nets = ref_import.run_reference_train(d, weight_seed=seed + 100, rng_seed=4242 + seed, batch_size=B,
                                                         num_samples=k, sampling_hops=hops, max_epochs=4,
                                                         eval_full_batch=False)
    st, recs = _oracle_epoch(d, seed, B, k, hops, {}, 4242 + seed, epochs=4)
    assert len(recs) == len(logs) == 16
    for r, l in zip(recs, logs):
        assert float(r["loss_c"]) == l["batch_loss_c"] and float(r["loss_gfn"]) == float(l["batch_loss_gfn"])
    assert logs[-1]["batch_loss_c"] < logs[0]["batch_loss_c"]                         # it trains
    o = rp.reference_evaluate(st, d.test_mask, full_batch=False, batch_size=B, stable_ties=False)
    assert o["f1"] == pytest.approx(test_f1, abs=1e-12)


@needs_reference
def test_oracle_embed_nodes_matches_live_reference_train(single_thread):
    """--embed_nodes (main.py:89-100,116; SURVEY.md section 8 row f4): the reference draws the table with nn.init.normal_
    from the global RNG, makes it an nn.Parameter inside optimizer_c and trains it.  Live ``train`` against the oracle with
    the same draw: per-batch losses bit-equal, the TABLE after the epoch equal to 1e-7 (dense Adam: rows of earlier batches
    keep moving), weights equal to 1e-7."""
    import torch.nn as nn
    name, seed, B, k, hops, dim = "tiny", 7, 32, 8, 2, 16
    rng_seed = 4242 + seed
    d_live = make_synth(name, seed=seed, features=False, F=dim)
    assert d_live.x is None and d_live.num_features == dim
    d_live.node_stores = [d_live]                         # main.py:99 `data.node_stores[0].x = embeddings`
    test_f1, logs, nets = ref_import.run_reference_train(d_live, weight_seed=seed + 100, rng_seed=rng_seed, batch_size=B,
                                                         num_samples=k, sampling_hops=hops, embed_nodes=True,
                                                         node_emb_dim=dim)
    assert isinstance(d_live.x, nn.Parameter) and tuple(d_live.x.shape) == (d_live.num_nodes, dim)
    # the oracle: same seed, same draw order (the table first, main.py:96-97, then the loader's base seed and the noise)
    d = make_synth(name, seed=seed, features=False, F=dim)
    torch.manual_seed(rng_seed)
    table = torch.FloatTensor(d.num_nodes, dim)
    nn.init.normal_(table)
    d.x = table
    st = rp.OracleState(d, sampling_hops=hops, num_samples=k, seed=seed + 100, dtype=torch.float32, embed_nodes=True)
    tr = d.train_mask.nonzero().squeeze(1)
    recs = [rp.reference_step(st, b[0], stable_ties=False)
            for b in torch.utils.data.DataLoader(torch.utils.data.TensorDataset(tr), batch_size=B)]
    assert len(recs) == len(logs)
    for r, l in zip(recs, logs):
        assert float(r["loss_c"]) == l["batch_loss_c"] and float(r["loss_gfn"]) == float(l["batch_loss_gfn"])
    assert not torch.equal(st.x.detach(), table)          # the table was trained ...
    assert torch.allclose(st.x.detach(), d_live.x.detach(), rtol=0, atol=1e-7 * float(table.abs().max()))   # ... identically
    ref_w, got_w = _flat_weights(nets), _flat_weights((st.gcn_c, st.gcn_gf, st.gcn_z))
    for key in ref_w:
        assert torch.allclose(got_w[key], ref_w[key], rtol=0, atol=1e-7 * float(ref_w[key].abs().max())), key


@needs_reference
def test_oracle_gcn_wiring_matches_live_reference_gcn_class(single_thread):
    """modules/gcn.py:9-42 imported live (oracle/ref_import.py::load_reference_gcn; GCNConv bound to the oracle's layer):
    the reference's own ``GCN`` -- layer list, ``edge_index[-i]`` for hidden layer i and ``edge_index[0]`` for the output
    layer when a list is given, relu / dropout placement, tuple return -- against ``OracleGCN`` on the same weights, for a
    single edge tensor, a per-layer list (2 and 3 layers) and in training mode with dropout (same RNG stream)."""
    g = torch.Generator().manual_seed(3)
    n, Fdim = 60, 9
    x = torch.randn(n, Fdim, generator=g)
    edges = [torch.randint(0, n, (2, m), generator=g) for m in (150, 90, 200)]
    for hidden, p in (([16, 4], 0.0), ([16, 8, 4], 0.0), ([16, 4], 0.5)):
        gen = torch.Generator().manual_seed(11)
        ref_mod = ref_import.load_reference_gcn(lambda in_channels, out_channels: rp.OracleGCNConv(in_channels, out_channels, gen))
        ref = ref_mod.GCN(Fdim, hidden_dims=hidden, dropout=p)
        mine = rp.OracleGCN(Fdim, hidden, dropout=p, generator=torch.Generator().manual_seed(11))
        assert [k for k, _ in ref.named_parameters()] == [k for k, _ in mine.named_parameters()]
        for (_, a), (_, b) in zip(ref.named_parameters(), mine.named_parameters()):
            assert torch.equal(a, b)
        for ei in (edges[0], edges[:len(hidden)]):
            for training in ((False, True) if p > 0 else (False,)):
                ref.train(training); mine.train(training)
                torch.manual_seed(5)
                a, mem = ref(x, ei)
                torch.manual_seed(5)
                b, _ = mine(x, ei)
                assert torch.equal(a, b) and isinstance(mem, float)


@needs_reference
def test_oracle_edge_cases_match_live_reference_utils():
    """Edge cases the domain has (SURVEY.md section 4): empty row lists, rows without neighbours, a self-loop, an empty
    column set, duplicated ids in the row list, one candidate, k = 1, k >= n -- the reference's own functions against the
    oracle's, bit for bit."""
    ru = ref_import.load_reference_utils()
    ei = torch.tensor([[0, 0, 1, 2, 4, 4, 6], [0, 2, 0, 1, 1, 2, 6]])           # nodes 3 and 5 have no out-edges; 0 and 6 loop
    N = 7
    adj_ref, adj = ref_import.reference_adjacency(ei, N), rp.build_adjacency(ei, N)
    empty = torch.tensor([], dtype=torch.long)
    for nodes in (empty, torch.tensor([3, 5]), torch.tensor([0, 3, 4]), torch.tensor([4, 0, 1, 2]), torch.tensor([6]),
                  torch.tensor([4, 4, 0])):
        a, b = ru.get_neighborhoods(nodes, adj_ref), rp.get_neighborhoods(nodes, adj)
        assert a.shape == b.shape and torch.equal(a, b), nodes
        for cols in (empty, torch.tensor([0, 1, 2]), torch.tensor([6, 2]), torch.arange(N)):
            a, b = ru.slice_adjacency(adj_ref, nodes, cols), rp.slice_adjacency(adj, nodes, cols)
            assert a.shape == b.shape and torch.equal(a, b), (nodes, cols)
    g = torch.Generator().manual_seed(0)
    for n, k in ((1, 1), (1, 4), (5, 1), (9, 9), (9, 8), (300, 299)):
        logits = torch.randn(n, 1, generator=g)
        nb = torch.arange(n) * 3 + 1
        torch.manual_seed(n * 31 + k)
        a = ru.sample_neighborhoods_from_probs(logits, nb, k)
        torch.manual_seed(n * 31 + k)
        b = rp.sample_neighborhoods_from_probs(logits, nb, k, stable_ties=False)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and a[2].keys() == b[2].keys(), (n, k)
        for key in a[2]:
            assert torch.equal(a[2][key], b[2][key]) or (torch.isnan(a[2][key]) and torch.isnan(b[2][key])), (n, k, key)
    # TensorMap: update / map round trip incl. re-update with another key set (stale entries stay, like the reference's)
    tm_a, tm_b = ru.TensorMap(size=N), rp.TensorMap(N)
    for keys in (torch.tensor([5, 2, 6]), torch.tensor([0, 6])):
        tm_a.update(keys); tm_b.update(keys)
        assert torch.equal(tm_a.map(torch.arange(N)[keys]), tm_b.map(torch.arange(N)[keys]))
        assert torch.equal(tm_a.values, tm_b.values)


@needs_reference
def test_host_side_dropins_inside_the_live_reference_loop(single_thread):
    """INTEGRATION.md section 1 (import-level drop-in), the part that needs no GPU: this repo's ``TensorMap`` and
    ``get_logger`` (grapes_b200/utils.py, pure torch / logging) bound in place of the reference's inside the reference's OWN
    ``train`` loop -- same losses on every batch, same weights, same score as the unmodified run."""
    from grapes_b200.utils import TensorMap, get_logger
    name, seed, B, k, hops = "tiny", 8, 32, 8, 2
    d = make_synth(name, seed=seed)
    kw = dict(weight_seed=seed + 100, rng_seed=4242 + seed, batch_size=B, num_samples=k, sampling_hops=hops, max_epochs=2,
              eval_full_batch=False)
    f1_a, logs_a, nets_a = ref_import.run_reference_train(d, **kw)
    f1_b, logs_b, nets_b = ref_import.run_reference_train(d, utils_overrides={"TensorMap": TensorMap, "get_logger": get_logger},
                                                          **kw)
    assert len(logs_a) == len(logs_b) == 8 and f1_a == f1_b
    for a, b in zip(logs_a, logs_b):
        assert a["batch_loss_c"] == b["batch_loss_c"] and float(a["batch_loss_gfn"]) == float(b["batch_loss_gfn"])
    for (ka, pa), (kb, pb) in zip(_flat_weights(nets_a).items(), _flat_weights(nets_b).items()):
        assert ka == kb and torch.equal(pa, pb)
