"""Shared checker of the whole-step parity tests: the device engine against the CPU oracle's restatement of
the reference's main.py:161-291 on the same graph, weights and injected Gumbel noise.

Bars (BASELINE.json north_star): frontier sets / dedup / relabel / blocks and sampled sets BIT-EXACT; logits,
aggregated features, losses and gradients within 1e-5 relative (fp32), measured against the oracle run in float64
and relative to each tensor's scale.

The relu kink.  A hidden unit whose layer-1 pre-activation is zero up to fp32 rounding can take the other relu branch
than the float64 oracle did (so can the reference's own fp32 run).  One such flip moves ONE row of that layer's weight
gradient by a finite amount.  The tcgen05 kernels keep their relu mask, so the check is explicit: every (node, unit)
whose branch differs from float64 must have |pre| < 1e-5 * max|pre| in the float64 oracle (a true kink), gradient rows
WITHOUT a verified flip hold the 1e-5 bar, and rows with one stay bounded."""
import torch

from oracle import reference_port as rp

TOL = 1e-5


def _rel(got, ref):
    ref = torch.as_tensor(ref).double()
    got = torch.as_tensor(got).double().cpu()
    return ((got - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item()


def _grad_tol(got32, ref64, floor=TOL):
    """Gradients are sums of O(frontier) signed terms; their fp32 conditioning is a property of the
    problem, not of the kernel.  Bar: 1e-5 relative, or -- when the reference's own fp32 evaluation
    (same path, CPU torch) is already further than that from float64 -- no worse than 2x the reference."""
    return max(floor, 2.0 * _rel(got32, ref64))


def _unpack_mask(mask_t: torch.Tensor, n: int) -> torch.Tensor:
    """maskT[(row group of 32)][D], bit r of word (g, d) = relu'(pre[32 g + r, d])  ->  bool [n, D]"""
    g = (n + 31) // 32
    w = mask_t[:g].cpu().to(torch.int64) & 0xffffffff
    bits = (w.unsqueeze(1) >> torch.arange(32, dtype=torch.int64).view(1, 32, 1)) & 1
    return bits.reshape(g * 32, -1)[:n].bool()


def relu_flips(eng, st, ref, weights_before):
    """Hidden units (rows of W1 / b1) of gcn_gf and gcn_z whose relu branch differs between the engine's tcgen05
    forward and the float64 oracle.  Asserts that every flipped entry is a kink.  Empty sets on the SIMT path."""
    flips = {"gcn_gf": set(), "gcn_z": set()}
    if not (eng.use_tc_bwd and not eng.random_sampling):
        return flips
    for h, b in enumerate(ref["hops"]):
        n = b["x"].shape[0]
        nets = [("gcn_gf", b["x"], eng.hops[h].mask_gf)]
        if h == 0:
            nets.append(("gcn_z", b["x"][:, :eng.F], eng.mask_z))
        for net, x, mask_t in nets:
            w = weights_before[net]
            pre = rp.gcn_conv(x.double(), b["local_neighborhoods"], w["gcn_layers.0.lin.weight"].double(),
                              w["gcn_layers.0.bias"].double())
            differ = _unpack_mask(mask_t, n) != (pre > 0)
            if differ.any():
                worst = pre[differ].abs().max().item()
                assert worst < 1e-5 * pre.abs().max().item(), \
                    f"hop {h} {net}: relu branch differs from float64 at |pre| = {worst:.3e} -- not a kink"
                flips[net] |= set(differ.nonzero()[:, 1].tolist())
    return flips


def _grad_ok(got, ref64, ref32, flipped_units, floor=TOL):
    """Elementwise bar on every row; rows (hidden units) with a VERIFIED relu-kink flip may exceed it, bounded."""
    tol = _grad_tol(ref32, ref64, floor)
    ref = torch.as_tensor(ref64).double()
    err = (torch.as_tensor(got).double().cpu() - ref).abs() / ref.abs().max().clamp_min(1e-30)
    if err.dim() > 1 and err.shape[0] == 1:
        err = err.reshape(-1)                                   # lin.weight of the width-1 output layer: one entry per unit
    rows = err.reshape(err.shape[0], -1).max(1).values if err.dim() > 1 else err
    bad = (rows > tol).nonzero().reshape(-1).tolist()
    if not set(bad) <= set(flipped_units):
        return False
    return bool(err.max() < 2e-2)


def well_separated(ref, ref32=None) -> bool:
    """True when the bit-exact sampled-set claim is meaningful for this draw: the k-th and (k+1)-th largest perturbed
    keys are further apart than fp32 rounding of the logits can move them, and the reference's own fp32 run selects the
    same sets as its float64 run."""
    for h in ref["hops"]:
        if h["keys"] is not None:
            srt = torch.sort(h["keys"], descending=True).values
            k = h["sampled"].numel()
            if not (srt[k - 1] - srt[k]) > 1e-4 * srt[:k + 1].abs().max():
                return False
    if ref32 is not None:
        for a, b in zip(ref32["hops"], ref["hops"]):
            if not torch.equal(a["sampled"], b["sampled"]):
                return False
    return True


def check_step(st, eng, targets, dev, apply_optim=True, post_optim=False, gumbel_noise=None):
    # first step: the 1e-5 bar.  After an Adam step the weights carry fp32 history (Adam divides by sqrt(v), which
    # amplifies the rounding noise of small gradient entries): floats are then held to the 1e-4 bar that
    # test_three_steps_with_adam holds the weights themselves to; integer contracts stay bit-exact.
    FT = 1e-4 if post_optim else TOL
    before = {k: {n: p.detach().clone() for n, p in net.named_parameters()}
              for k, net in (("gcn_gf", st.gcn_gf), ("gcn_z", st.gcn_z))}
    ref = rp.reference_step(st, targets, gumbel_noise=gumbel_noise, apply_optim=apply_optim)
    ref32 = rp.reference_step(st.fp32, targets, gumbel_noise=[h["noise"] for h in ref["hops"]], apply_optim=apply_optim)
    for a, b in zip(ref32["hops"], ref["hops"]):
        assert torch.equal(a["sampled"], b["sampled"]), "fp32 / fp64 oracle disagree on the sampled set: pick another seed"
    for h in ref["hops"]:                     # the selection must be well separated for a bit-exact set claim
        if h["keys"] is not None:
            srt = torch.sort(h["keys"], descending=True).values
            k = h["sampled"].numel()
            assert (srt[k - 1] - srt[k]) > 1e-4 * srt[:k + 1].abs().max(), "pick another seed: top-k boundary too tight"
    noise = [None if h["noise"] is None else h["noise"].float().to(dev) for h in ref["hops"]]
    rec = eng.step(targets.to(dev), gumbel_noise=noise, apply_optim=apply_optim, record=True)
    eng.check_overflow()
    for h, (a, b) in enumerate(zip(rec["hops"], ref["hops"])):
        # ---- integer contracts: bit-exact ----
        assert torch.equal(a["prev"].cpu().long(), b["prev"]), f"hop {h} prev"
        assert torch.equal(a["batch_nodes"].cpu().long(), b["batch_nodes"]), f"hop {h} batch_nodes"
        assert torch.equal(a["neighbor_nodes"].cpu().long(), b["neighbor_nodes"]), f"hop {h} neighbor_nodes"
        assert torch.equal(a["nb_local"].cpu().long(), b["nb_local"]), f"hop {h} nb_local"
        loc = torch.stack([a["e_src"], a["e_dst"]]).cpu().long()
        assert torch.equal(loc, b["local_neighborhoods"]), f"hop {h} local edges"
        glob = torch.stack([a["prev"].long()[a["e_row"].long()], a["e_col"].long()]).cpu()
        assert torch.equal(glob, b["neighborhoods"]), f"hop {h} neighborhoods"
        assert torch.equal(a["block_edges"].cpu().long(), b["block_edges"]), f"hop {h} block edges"
        assert torch.equal(a["sampled"].cpu().long(), b["sampled"]), f"hop {h} sampled set"
        # ---- floating point: 1e-5 relative ----
        if not st.random_sampling:
            ei, w = rp.gcn_norm(b["local_neighborhoods"], b["x"].shape[0], dtype=torch.float64)
            y_ref = torch.zeros_like(b["x"]).index_add(0, ei[1], b["x"][ei[0]] * w.unsqueeze(1))
            assert _rel(a["Y"][:, :y_ref.shape[1]], y_ref) < FT, f"hop {h} aggregated features"
            assert _rel(a["logits_all"], b["logits_all"]) < FT, f"hop {h} logits"
        assert _rel(a["log_prob"], b["log_prob"]) < FT, f"hop {h} log_prob"
        if b["stats"]:
            for i, key in enumerate(("min_prob", "max_prob", "mean_entropy", "std_entropy")):
                assert abs(a["stats"][i].item() - b["stats"][key].item()) < 1e-4 * max(1.0, abs(b["stats"][key].item()))
    assert torch.equal(rec["all_nodes"].cpu().long(), ref["all_nodes"])
    assert torch.equal(rec["target_local"].cpu().long(), ref["local_target_ids"])
    assert torch.equal(rec["cl_edges"][0].cpu().long(), ref["edge_indices"][-1])
    assert torch.equal(rec["cl_edges"][1].cpu().long(), ref["edge_indices"][0])
    assert _rel(rec["logits_c"], ref["logits_c"]) < FT
    s = rec["scalars"]
    assert abs(s["loss_c"] - ref["loss_c"].item()) < FT * abs(ref["loss_c"].item())
    assert abs(s["tot_log_prob"] - ref["tot_log_prob"].item()) < FT * abs(ref["tot_log_prob"].item())
    for name, gref in ref["grads_c"].items():
        assert _grad_ok(rec["grads"]["gcn_c"][name], gref, ref32["grads_c"][name], (), FT), f"grad gcn_c {name}"
    if not st.random_sampling:
        flips = relu_flips(eng, st, ref, before)
        rec["relu_flips"] = flips
        assert abs(s["log_z"] - ref["log_z"].item()) < FT * max(1.0, abs(ref["log_z"].item()))
        assert abs(s["loss_gfn"] - ref["loss_gfn"].item()) < 4 * FT * abs(ref["loss_gfn"].item())
        for name, gref in ref["grads_gf"].items():
            assert _grad_ok(rec["grads"]["gcn_gf"][name], gref, ref32["grads_gf"][name], flips["gcn_gf"], FT), \
                f"grad gcn_gf {name} (units with a verified kink flip: {sorted(flips['gcn_gf'])})"
        for name, gref in ref["grads_z"].items():
            if gref is not None:
                assert _grad_ok(rec["grads"]["gcn_z"][name], gref, ref32["grads_z"][name], flips["gcn_z"], FT), \
                    f"grad gcn_z {name} (units with a verified kink flip: {sorted(flips['gcn_z'])})"
    return rec, ref
