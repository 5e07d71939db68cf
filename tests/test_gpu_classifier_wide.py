"""The classifier half of a training step in its "wide" form, taken when cap_A = B + H * k exceeds
GrapesEngine.PREP_MAX_ROWS (4096): grapes_relabel + grapes_build_csr instead of the one-launch grapes_classifier_prep,
and the target-row loss (k_loss_rows + k_loss_final, then grapes_colsum for the bias-2 gradient) instead of the
row-parallel one.  Users reach it with --batch_size 4096 or --num_samples 2048.

  - the two forms on the same step: every integer output, the logits, the hidden layer, d loss / d logits and the
    gcn_c weight gradients bit for bit; the reductions they order differently at 1e-6;
  - the wide form with more than 4096 live rows (40 000-node graph, cap_A 4608 and 9728) against the float64 oracle at
    the bars of tests/parity_utils.py: cross-entropy and multilabel, reg_param, REINFORCE, learned node features,
    dropout, tensor cores, three Adam steps, CUDA-graph replay;
  - mini-batch evaluation (GrapesEngine.predict) with batches of 4200 targets.

Each test asserts the form it exercises (cap_A against PREP_MAX_ROWS, and the GEMM tile form from the device's SM count
with the dispatch rule of grapes_gemm), so a later threshold change cannot quietly turn it into a duplicate."""
import contextlib
import math

import pytest
import torch

from dropout_utils import engine_masks, replay_masks
from oracle import reference_port as rp
from parity_utils import TOL, _rel, check_step, well_separated
from test_gpu_engine import _setup

pytestmark = pytest.mark.gpu

MID = dict(N=40_000, E_dir=1_200_000, F=100, C=47, n_train=30_000, num_samples=256, sampling_hops=2)


def _big_tiles(eng, N):
    """True when grapes_gemm takes the 128 x 128 tiles for a [cap_A x N] product on this device"""
    sms = torch.cuda.get_device_properties(eng.device).multi_processor_count
    return math.ceil(N / 128) * math.ceil(eng.cap_A / 128) >= sms


def _mid_setup(batch_size, seed, dev, **kw):
    """test_gpu_engine._setup on the 40 000-node graph with a temporary SHAPES entry"""
    from grapes_b200.synth import SHAPES
    SHAPES["mid_wide"] = dict(MID, batch_size=batch_size)
    try:
        return _setup("mid_wide", seed, dev, **kw)
    finally:
        SHAPES.pop("mid_wide")


def _draw(st, train_idx, B, start):
    """the first full batch from `start` on whose top-k boundaries are well separated in the float64 and fp32 oracles
    (the attempt loop of test_gpu_parity_fullsize); returns (targets, noise, next start)"""
    for a in range(start, train_idx.numel() // B):
        targets = train_idx[a * B:(a + 1) * B]
        pre = rp.reference_step(st, targets, apply_optim=False)
        noise = [h["noise"] for h in pre["hops"]]
        if well_separated(pre, rp.reference_step(st.fp32, targets, gumbel_noise=noise, apply_optim=False)):
            return targets, noise, a + 1
    pytest.fail(f"no well-separated draw in batches {start}..{train_idx.numel() // B - 1}")


# ---------------------------------------------------------------------------------------------------------------------
def test_prep_and_wide_forms_agree(cuda_device):
    """The same step (small graph, seed 1, same targets and injected noise) through both forms."""
    dev = cuda_device
    d, st, prep, train_idx, B = _setup("small", 1, dev)
    _, _, wide, _, _ = _setup("small", 1, dev)
    wide.PREP_MAX_ROWS = 0
    assert prep.cap_A <= prep.PREP_MAX_ROWS and wide.cap_A > wide.PREP_MAX_ROWS
    gen = torch.Generator(device=dev).manual_seed(8)
    noise = [torch.rand(prep.cap_n, generator=gen, device=dev).clamp_(1e-7, 1 - 1e-7).log().neg().log().neg()
             for _ in range(prep.H)]
    t = train_idx[:B].to(dev)
    recs = []
    for eng in (prep, wide):
        rec = eng.step(t, gumbel_noise=noise, apply_optim=False, record=True)
        eng.check_overflow()
        A = eng.count("A")
        rec["hidden_c"] = eng.out1[:A].clone()
        rec["dlogits"] = eng.dlogits[:A].clone()
        recs.append(rec)
    a, b = recs
    for h, (ha, hb) in enumerate(zip(a["hops"], b["hops"])):
        for key in ("prev", "batch_nodes", "neighbor_nodes", "sampled", "block_edges"):
            assert torch.equal(ha[key], hb[key]), f"hop {h} {key}"
    for key in ("all_nodes", "target_local", "logits_c", "hidden_c", "dlogits"):
        assert torch.equal(a[key], b[key]), key
    for e1, e2 in zip(a["cl_edges"], b["cl_edges"]):
        assert torch.equal(e1, e2)
    gc_a, gc_b = a["grads"]["gcn_c"], b["grads"]["gcn_c"]
    for name in ("gcn_layers.0.lin.weight", "gcn_layers.0.bias", "gcn_layers.1.lin.weight"):
        assert torch.equal(gc_a[name], gc_b[name]), name
    # the loss sums over A rows (prep) or over the B target rows (wide); the bias-2 column sums come from the loss
    # launch or from grapes_colsum: differently ordered reductions
    assert _rel(gc_b["gcn_layers.1.bias"], gc_a["gcn_layers.1.bias"].cpu()) < 1e-6
    for k in ("loss_c", "loss_gfn"):
        assert abs(a["scalars"][k] - b["scalars"][k]) <= 1e-6 * abs(a["scalars"][k]), k
    for net in ("gcn_gf", "gcn_z"):
        for name, g in a["grads"][net].items():
            assert _rel(b["grads"][net][name], g.cpu()) < 1e-6, f"{net} {name}"


# ---------------------------------------------------------------------------------------------------------------------
# The classifier kernels are the same on both engines; the engine choice only changes the sampler nets.  On this
# 40 000-row frontier (10 M sampler pre-activations) a unit whose pre-activation is zero up to fp32 rounding is likely,
# and the SIMT sampler backward keeps no relu mask, so check_step cannot verify such a flip: the SIMT trajectory-balance
# step of seed 1 misses the 1e-5 bar on one gcn_z bias entry for that reason.  The default engine (tensor cores) records
# the mask and every flip is verified against float64, so the cases whose sampler gradients carry the full
# trajectory-balance scale run on it; the SIMT engine keeps three cases.
TC = {"use_tensor_cores": True}
WIDE = {                            # name -> (batch size, seed, engine / oracle arguments)
    "tb_tensor_cores": (4096, 2, TC),
    "simt_multilabel": (4096, 3, {"multilabel": True}),
    "simt_reg_param": (4096, 4, {"reg_param": 0.1}),
    "simt_reinforce": (4096, 5, {"reinforce_baseline": True}),
    "embed_nodes": (4096, 6, dict(TC, embed_nodes=True)),
    "dropout": (4096, 7, dict(TC, dropout=0.5)),
    "big_tiles": (9216, 8, TC),
}


@pytest.mark.parametrize("case", list(WIDE))
def test_wide_step_parity(cuda_device, case):
    """One step with more than 4096 live rows against the float64 oracle.  cap_A 4608 (B 4096, k 256, 2 hops) takes the
    64 x 64 GEMM tiles on a B200; cap_A 9728 (B 9216) the 128 x 128 tiles for the W1 forward and dZ W2 gated."""
    dev = cuda_device
    B, seed, kw = WIDE[case]
    p = kw.get("dropout", 0.0)
    d, st, eng, train_idx, B = _mid_setup(B, seed, dev, **kw)
    assert eng.cap_A > eng.PREP_MAX_ROWS
    assert _big_tiles(eng, eng.D) == (case == "big_tiles")
    with replay_masks(engine_masks(seed, 0, p)) if p else contextlib.nullcontext():
        targets, noise, _ = _draw(st, train_idx, B, 0)
        rec, ref = check_step(st, eng, targets, dev, apply_optim=False, gumbel_noise=noise)
    A = rec["all_nodes"].numel()
    assert A > 4096, f"only {A} live rows"
    if kw.get("embed_nodes"):
        assert _rel(rec["grad_x_rows"], ref["grad_x"][ref["all_nodes"]]) < TOL
    if p:
        k1, k2 = rec["dropout_keep"]
        assert 0 < k1.float().mean() < 1 and not rec["logits_c"][~k2].any()


def test_wide_three_adam_steps(cuda_device):
    """Three steps with both optimisers on the wide form (post-optimiser bar 1e-4 from the second step on)."""
    dev = cuda_device
    d, st, eng, train_idx, B = _mid_setup(4096, 9, dev)
    assert eng.cap_A > eng.PREP_MAX_ROWS and not _big_tiles(eng, eng.D)
    start = 0
    for i in range(3):
        targets, noise, start = _draw(st, train_idx, B, start)
        check_step(st, eng, targets, dev, apply_optim=True, post_optim=(i > 0), gumbel_noise=noise)
    assert eng.adam_steps.tolist() == [3.0, 3.0]


def test_wide_graph_replay_matches_eager(cuda_device):
    """Captured CUDA-graph replay of the wide form equals eager launches bit for bit (losses, all_nodes, Philox state,
    gradients, weights, Adam moments), two steps."""
    dev = cuda_device
    d, _, eng, train_idx, B = _mid_setup(4096, 10, dev)
    _, _, eng2, _, _ = _mid_setup(4096, 10, dev)
    assert eng.cap_A > eng.PREP_MAX_ROWS
    for i in range(2):
        t = train_idx[i * B:(i + 1) * B].to(dev)
        eng.step(t, use_graph=False)
        eng2.step(t, use_graph=True)
        torch.cuda.synchronize()
        assert torch.equal(eng.scal, eng2.scal), f"step {i}: losses differ between eager and graph replay"
        assert torch.equal(eng.all_nodes, eng2.all_nodes)
    eng.check_overflow(); eng2.check_overflow()
    assert eng2.count("A") > 4096
    for name in ("rng_state", "grads", "params", "exp_avg_sq"):
        assert torch.equal(getattr(eng, name), getattr(eng2, name)), name


def test_wide_mini_batch_eval(cuda_device):
    """GrapesEngine.predict with batches of 4200 targets (cap_A 4712, the last batch partial) against the oracle's
    mini-batch evaluation: per-hop candidates, top-k sets and blocks bit-exact, logits at 1e-5, predictions equal."""
    from grapes_b200.engine import GrapesEngine
    from grapes_b200.synth import SHAPES
    import test_gpu_eval as E
    dev, bs = cuda_device, 4200
    SHAPES["mid_wide"] = dict(MID, batch_size=bs)
    try:
        cfg, d, st, g, _, _, _ = E._setup("mid_wide", 11, dev)
    finally:
        SHAPES.pop("mid_wide")
    mask = d.val_mask
    idx = mask.nonzero().squeeze(1)
    assert idx.numel() % bs != 0
    ref = rp.reference_evaluate(st, mask, full_batch=False, batch_size=bs)
    eng = GrapesEngine(g, d.x.to(dev), d.y.to(dev), num_classes=d.num_classes, batch_size=bs,
                       num_samples=cfg["num_samples"], sampling_hops=cfg["sampling_hops"], use_tensor_cores=False)
    eng.load_state_dicts(gcn_c=st.gcn_c.state_dict(), gcn_gf=st.gcn_gf.state_dict())
    assert eng.cap_A > eng.PREP_MAX_ROWS
    out = torch.zeros(bs, dtype=torch.int32, device=dev)
    preds = []
    for bi, t in enumerate(torch.split(idx, bs)):
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
            assert torch.equal(blk, rh["block_edges"]), f"batch {bi} hop {h}: block"
        A = eng.count("A")
        assert torch.equal(eng.all_nodes[:A].cpu().long(), rb["all_nodes"])
        E._close(eng.logits_c[:A], rb["logits"])
        preds.append(out[:b].cpu().long().clone())
    assert len(preds) == 2 and preds[-1].numel() < bs
    assert torch.equal(torch.cat(preds), ref["predictions"])
