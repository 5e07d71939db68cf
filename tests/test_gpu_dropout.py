"""Dropout in the classifier GCN of the device training step (``--dropout p``; modules/gcn.py:33,37, main.py:107-112).

The engine's masks are a pure function of (seed, step, rank, site, row, col) (tests/dropout_utils.py restates it in
numpy).  The parity tests replay exactly those masks inside the float64 oracle (dropout_utils.replay_masks) and hold the
step to the bars of tests/parity_utils.py; the recorded masks must equal the numpy ones bit for bit, and the kernels'
outputs must be zero wherever an entry was dropped."""
import math

import numpy as np
import pytest
import torch

from dropout_utils import engine_masks, keep_mask, replay_masks, tag, threshold
from oracle import reference_port as rp
from parity_utils import TOL, _rel, check_step, well_separated
from test_gpu_engine import _setup

pytestmark = pytest.mark.gpu


def _check_masks(eng, rec, seed, step, rank=0):
    """recorded masks == numpy restatement; dropped entries of the hidden layer and of the logits are exactly zero"""
    A = rec["all_nodes"].numel()
    k1, k2 = rec["dropout_keep"]
    thr = threshold(eng.dropout)
    assert rec["dropout_step"] == step
    assert np.array_equal(k1.cpu().numpy(), keep_mask(seed, step, tag(0, rank), thr, A, eng.D)), "hidden-layer mask"
    assert np.array_equal(k2.cpu().numpy(), keep_mask(seed, step, tag(1, rank), thr, A, eng.C)), "logits mask"
    assert not rec["hidden_c"][~k1].any() and not rec["logits_c"][~k2].any()
    return k1, k2


PARITY = {                                  # name -> (graph, seed, p, extra arguments)
    "ce_p0.1": ("tiny", 0, 0.1, {}),
    "ce_p0.5": ("small", 1, 0.5, {}),
    "multilabel": ("tiny", 6, 0.5, {"multilabel": True}),
    "reg_param": ("tiny", 5, 0.5, {"reg_param": 0.1}),
    "embed_nodes": ("tiny", 0, 0.5, {"embed_nodes": True}),
}


@pytest.mark.parametrize("case", sorted(PARITY))
def test_step_parity_with_dropout(cuda_device, case):
    """One step against the float64 oracle with the device's masks replayed: logits_c (after dropout), loss_c, the
    three gradient sets and loss_gfn at the bars of every other step test (target-row loss form, cap_A <= 4096)."""
    name, seed, p, kw = PARITY[case]
    d, st, eng, train_idx, B = _setup(name, seed, cuda_device, dropout=p, **kw)
    assert eng.cap_A <= 4096
    with replay_masks(engine_masks(seed, 0, p)):
        rec, ref = check_step(st, eng, train_idx[:B], cuda_device, apply_optim=False)
    k1, k2 = _check_masks(eng, rec, seed, 0)
    assert 0 < k1.float().mean() < 1 and 0 < k2.float().mean() < 1
    if kw.get("embed_nodes"):
        an = ref["all_nodes"]
        assert _rel(rec["grad_x_rows"], ref["grad_x"][an]) < TOL


def test_step_parity_with_dropout_arxiv_shape(cuda_device):
    """The BASELINE arxiv-shaped graph on the default path (tcgen05 sampler GEMMs, multi-stream step), p = 0.5."""
    import scipy.sparse as sp
    from bench import build_workload
    from grapes_b200.engine import GrapesEngine
    from grapes_b200.graph import DeviceGraph
    from grapes_b200.synth import SynthData
    dev, p = cuda_device, 0.5
    torch.manual_seed(4242)
    cfg, indptr, indices, x, y, train_idx = build_workload("arxiv", 0, dev, native_csr=True)
    N, B = cfg["N"], cfg["batch_size"]
    ip, ix = indptr.cpu().numpy(), indices.cpu().numpy()
    adj = sp.csr_matrix((np.ones(ix.shape[0], dtype=bool), ix, ip), shape=(N, N))
    data = SynthData(x=x.cpu(), y=y.cpu(), edge_index=torch.zeros(2, 0, dtype=torch.long), train_mask=None,
                     val_mask=None, test_mask=None, num_nodes=N, num_features=cfg["F"], num_classes=cfg["C"])
    kw = dict(sampling_hops=cfg["sampling_hops"], num_samples=cfg["num_samples"], hidden_dim=256, seed=100,
              adjacency=adj, dropout=p)
    st = rp.OracleState(data, dtype=torch.float64, **kw)
    st.fp32 = rp.OracleState(data, dtype=torch.float32, **kw)
    eng = GrapesEngine(DeviceGraph(indptr, indices, N), x, y, num_classes=cfg["C"], batch_size=B,
                       num_samples=cfg["num_samples"], sampling_hops=cfg["sampling_hops"], hidden_dim=256, seed=0,
                       dropout=p)
    assert eng.use_tc and eng.multi_stream
    eng.load_state_dicts(gcn_c=st.gcn_c.state_dict(), gcn_gf=st.gcn_gf.state_dict(), gcn_z=st.gcn_z.state_dict())
    with replay_masks(engine_masks(0, 0, p)):
        for attempt in range(6):
            targets = train_idx[(5 + attempt) * B:(6 + attempt) * B].cpu()
            pre = rp.reference_step(st, targets, apply_optim=False)
            noise = [h["noise"] for h in pre["hops"]]
            if well_separated(pre, rp.reference_step(st.fp32, targets, gumbel_noise=noise, apply_optim=False)):
                break
        else:
            pytest.fail("no well-separated draw in 6 batches")
        rec, ref = check_step(st, eng, targets, dev, apply_optim=False, gumbel_noise=noise)
    _check_masks(eng, rec, 0, 0)


def test_masks_and_loss_of_the_wide_form(cuda_device):
    """cap_A > 4096 takes the other loss form (k_loss_rows / k_loss_final): masks bit for bit, the dropped logits zero,
    loss_c and d loss / d b2 against float64 autograd on the recorded dropped logits."""
    from grapes_b200.engine import GrapesEngine
    from grapes_b200.graph import DeviceGraph
    from grapes_b200.synth import make_synth
    p, reg = 0.5, 0.1
    d = make_synth("small", seed=1)
    eng = GrapesEngine(DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=cuda_device), d.x.to(cuda_device),
                       d.y.to(cuda_device), num_classes=d.num_classes, batch_size=1100, num_samples=1024,
                       sampling_hops=3, reg_param=reg, seed=1, dropout=p)
    assert eng.cap_A > 4096
    t = d.train_mask.nonzero().squeeze(1)[:1100]
    rec = eng.step(t.to(cuda_device), apply_optim=False, record=True)
    eng.check_overflow()
    _, k2 = _check_masks(eng, rec, 1, 0)
    l = rec["logits_c"].double().cpu().requires_grad_(True)
    tl = rec["target_local"].cpu().long()
    loss = torch.nn.functional.cross_entropy(l[tl], d.y[t]) + reg * torch.var(l, dim=1).sum()
    loss.backward()
    db2 = (l.grad * k2.cpu().double() / (1 - p)).sum(0)
    assert abs(rec["scalars"]["loss_c"] - loss.item()) < TOL * abs(loss.item())
    assert _rel(rec["grads"]["gcn_c"]["gcn_layers.1.bias"], db2) < TOL


def test_three_adam_steps_with_dropout(cuda_device):
    """Three steps with both optimisers against the oracle, each step with that step's masks (post-optimiser bar 1e-4)."""
    p, seed = 0.5, 2
    d, st, eng, train_idx, B = _setup("cora", seed, cuda_device, dropout=p)
    nsteps = 3
    for i in range(nsteps):
        with replay_masks(engine_masks(seed, i, p)):
            rec, _ = check_step(st, eng, train_idx[i * B:(i + 1) * B], cuda_device, apply_optim=True,
                                post_optim=(i > 0))
        _check_masks(eng, rec, seed, i)
    for key, net, net32, lr in (("gcn_c", st.gcn_c, st.fp32.gcn_c, 1e-3), ("gcn_gf", st.gcn_gf, st.fp32.gcn_gf, 1e-4),
                                ("gcn_z", st.gcn_z, st.fp32.gcn_z, 1e-4)):
        for (name, w), (_, w32) in zip(net.named_parameters(), net32.named_parameters()):
            ref = w.detach().double()
            err = (eng.state_dicts()[key][name].double().cpu() - ref).abs()
            assert err.max() <= 2.0 * lr * nsteps * 1.01, f"{key} {name}: beyond the Adam sign-flip bound"
            scale = ref.abs().max().clamp_min(1e-30)
            frac = (err > 1e-4 * scale).double().mean().item()
            frac32 = ((w32.detach().double() - ref).abs() > 1e-4 * scale).double().mean().item()
            assert frac <= max(0.01, 3.0 * frac32), f"{key} {name}: {frac:.4f} of the weights off by > 1e-4"


def test_consecutive_steps_draw_new_masks_and_leave_the_sampler_alone(cuda_device):
    """Every step advances the mask counter once, with and without the optimiser; the sampler's Philox stream and the
    first step's sampled sets are those of an engine without dropout."""
    d, st, eng, train_idx, B = _setup("small", 1, cuda_device, dropout=0.5)
    _, _, eng0, _, _ = _setup("small", 1, cuda_device)
    masks = []
    for i, opt in enumerate((True, False, False, True)):
        t = train_idx[i * B:(i + 1) * B].to(cuda_device)
        r = eng.step(t, apply_optim=opt, record=True)
        r0 = eng0.step(t, apply_optim=opt, record=True)
        k1, _ = _check_masks(eng, r, 1, i)
        masks.append(k1)
        if i == 0:
            for h, (a, b) in enumerate(zip(r["hops"], r0["hops"])):
                assert torch.equal(a["sampled"], b["sampled"]), f"hop {h}"
    assert int(eng.drop_state[1]) == 4 and int(eng0.drop_state[1]) == 0
    torch.cuda.synchronize()
    assert torch.equal(eng.rng_state, eng0.rng_state)
    for a, b in zip(masks, masks[1:]):
        m = min(a.shape[0], b.shape[0])
        assert (a[:m] != b[:m]).float().mean() > 0.3


def test_graph_replay_and_prefetch_match_eager(cuda_device):
    """CUDA-graph replay with and without the next batch's prefetched front end equals eager steps bit for bit; the
    dropout forms replace their plain counterparts, so the graph has the launch count of an engine without dropout."""
    engines = [_setup("cora", 0, cuda_device, dropout=0.5)[2] for _ in range(3)]
    d, _, plain, train_idx, B = _setup("cora", 0, cuda_device)
    _, _, zero, _, _ = _setup("cora", 0, cuda_device, dropout=0.0)
    batches = [train_idx[i * B:(i + 1) * B].to(torch.int32).to(cuda_device).contiguous() for i in range(3)]
    for i, t in enumerate(batches):
        nxt = batches[i + 1] if i + 1 < len(batches) else None
        engines[0].step(t)
        engines[1].step(t, use_graph=True)
        engines[2].step(t, use_graph=True, next_targets=nxt)
        plain.step(t, use_graph=True)
        zero.step(t, use_graph=True)
    torch.cuda.synchronize()
    e0 = engines[0]
    for e in engines[1:]:
        e.check_overflow()
        for name in ("params", "grads", "exp_avg_sq", "rng_state", "drop_state", "scal"):
            assert torch.equal(getattr(e0, name), getattr(e, name)), name
    assert int(e0.drop_state[1]) == 3
    assert zero.launches_per_graph == plain.launches_per_graph == engines[1].launches_per_graph
    assert torch.equal(zero.params, plain.params)


def test_p_one_drops_everything(cuda_device):
    d, st, eng, train_idx, B = _setup("tiny", 0, cuda_device, dropout=1.0)
    rec = eng.step(train_idx[:B].to(cuda_device), apply_optim=False, record=True)
    s = rec["scalars"]
    assert all(math.isfinite(v) for v in s.values())
    assert not rec["logits_c"].any() and not rec["dropout_keep"][0].any() and not rec["dropout_keep"][1].any()
    for name, g in rec["grads"]["gcn_c"].items():
        assert not g.any(), name
    assert abs(s["loss_c"] - math.log(d.num_classes)) < 1e-5 * math.log(d.num_classes)
    assert all(torch.isfinite(g).all() for net in rec["grads"].values() for g in net.values())


def test_evaluation_never_drops(cuda_device):
    """predict / evaluate (full batch and mini-batch) of an engine with p = 0.5 equal those of an engine without dropout
    holding the same weights, bit for bit."""
    from grapes_b200.train import evaluate
    d, _, eng, train_idx, B = _setup("small", 1, cuda_device, dropout=0.5)
    _, _, eng0, _, _ = _setup("small", 1, cuda_device)
    eng.step(train_idx[:B].to(cuda_device))
    sd = eng.state_dicts()
    eng0.load_state_dicts(gcn_c=sd["gcn_c"], gcn_gf=sd["gcn_gf"], gcn_z=sd["gcn_z"])
    tgt = d.test_mask.nonzero().squeeze(1)[:B].to(torch.int32).to(cuda_device)
    outs = []
    for e in (eng, eng0):
        o = torch.zeros(B, dtype=torch.int32, device=cuda_device)
        e.predict(tgt, o)
        torch.cuda.synchronize()
        outs.append(o)
    assert torch.equal(outs[0], outs[1])
    for full in (True, False):
        assert evaluate(eng, d, d.test_mask, full_batch=full) == evaluate(eng0, d, d.test_mask, full_batch=full)


def test_train_with_dropout_runs(cuda_device):
    from grapes_b200.args import Arguments
    from grapes_b200.synth import make_synth
    from grapes_b200.train import train
    a = Arguments()
    a.dataset, a.max_epochs, a.batch_size, a.num_samples, a.sampling_hops = "tiny", 2, 32, 8, 2
    a.eval_frequency, a.dropout = 1, 0.5
    d = make_synth("tiny", seed=0)
    logs = []
    f1, *_ = train(a, data=d, device=cuda_device, step_log=logs.append)
    assert len(logs) == 2 * 4 and all(math.isfinite(v) for log in logs for v in log.values())
    assert 0.0 <= f1 <= 1.0 and train.last_engine.dropout == 0.5 and int(train.last_engine.drop_state[1]) == 8
    a.dropout = 1.5
    with pytest.raises(ValueError, match="dropout probability has to be between 0 and 1"):
        train(a, data=make_synth("tiny", seed=0), device=cuda_device)
