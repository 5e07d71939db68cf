"""Whole-step parity of the device-resident engine with the CPU oracle's restatement of
main.py:161-291 (SURVEY.md section 8 rows a2-a13) on the same synthetic graphs, same initial
weights and the same injected Gumbel noise.

Bars (BASELINE.json north_star): frontier sets / dedup / relabel / blocks and sampled sets
BIT-EXACT; logits, aggregated features, losses and gradients within 1e-5 relative (fp32),
measured against the oracle run in float64 and relative to each tensor's scale."""
import pytest
import torch

from grapes_b200.synth import make_synth
from oracle import reference_port as rp
from parity_utils import TOL, _rel, check_step as _check_step

pytestmark = pytest.mark.gpu


def _setup(name, seed, dev, use_tensor_cores=False, **kw):
    """use_tensor_cores=False: the fp32 SIMT kernels, whose rounding is at the reference's own level, so the strict
    1e-5 bars apply elementwise.  The tcgen05 (3xTF32) path is covered by test_tensor_core_engine_* below."""
    from grapes_b200.engine import GrapesEngine
    from grapes_b200.graph import DeviceGraph
    from grapes_b200.synth import SHAPES
    cfg = dict(SHAPES[name])
    torch.manual_seed(1000 + seed)     # the oracle draws its Gumbel noise from the global CPU generator
    over = {"F": kw.pop("F")} if "F" in kw else {}
    d = make_synth(name, seed=seed, multilabel=kw.pop("multilabel", False), power_law=kw.pop("power_law", 0.0), **over)
    feature_bf16 = kw.pop("feature_bf16", False)
    if feature_bf16:                     # the table is STORED in bf16; the oracle computes on exactly those values
        d.x = d.x.bfloat16().float()
    eng_kw = {k: kw.pop(k) for k in ("cap_nodes", "cap_edges", "cap_block", "multi_stream") if k in kw}   # engine only
    hp = dict(sampling_hops=cfg["sampling_hops"], num_samples=cfg["num_samples"])
    hp.update(kw)
    hidden = hp.pop("hidden_dim", 256)
    st = rp.OracleState(d, seed=seed + 100, dtype=torch.float64, hidden_dim=hidden, **hp)
    # the same reference path in its own precision (fp32): measures how far fp32 itself sits from fp64
    st.fp32 = rp.OracleState(d, seed=seed + 100, dtype=torch.float32, hidden_dim=hidden, **hp)
    g = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=dev)
    eng = GrapesEngine(g, d.x.to(dev).bfloat16() if feature_bf16 else d.x.to(dev), d.y.to(dev),
                       num_classes=d.num_classes, batch_size=cfg["batch_size"],
                       hidden_dim=st.gcn_c.gcn_layers[0].lin.weight.shape[0],
                       lr_gc=1e-3, lr_gf=1e-4, seed=seed, use_tensor_cores=use_tensor_cores, **eng_kw, **hp)
    eng.load_state_dicts(gcn_c=st.gcn_c.state_dict(), gcn_gf=st.gcn_gf.state_dict(), gcn_z=st.gcn_z.state_dict())
    train_idx = d.train_mask.nonzero().squeeze(1)
    return d, st, eng, train_idx, cfg["batch_size"]


@pytest.mark.parametrize("name,seed", [("tiny", 0), ("cora", 0), ("small", 1)])
def test_step_parity_trajectory_balance(cuda_device, name, seed):
    d, st, eng, train_idx, B = _setup(name, seed, cuda_device)
    _check_step(st, eng, train_idx[:B], cuda_device, apply_optim=False)


@pytest.mark.parametrize("F,use_tc", [(38, False), (41, True), (602, True)])
def test_step_parity_feature_width_not_multiple_of_4(cuda_device, F, use_tc):
    """Reddit has 602 features, Cora 1433: the engine re-pitches the table to ldx = round_up(F, 4) and the TMA-staged
    aggregation (frontier >= 4096 rows here) carries a partial last feature lane.  Same bars as every other step test."""
    d, st, eng, train_idx, B = _setup("small", 1, cuda_device, use_tensor_cores=use_tc, F=F)
    assert eng.ldx == (F + 3) // 4 * 4 and eng.cap_n >= 4096 and tuple(eng.x.shape) == (d.num_nodes, F)
    _check_step(st, eng, train_idx[:B], cuda_device, apply_optim=False)


@pytest.mark.parametrize("use_tc", [False, True])
def test_step_parity_power_law_hub_rows(cuda_device, use_tc):
    """SURVEY.md section 8(d) stress variant: Zipf-like endpoints -> a few hub rows with thousands of entries next to
    isolated nodes (hub worklist of the per-row sort, long rows in the expansion, skewed in-degrees in gcn_norm)."""
    d, st, eng, train_idx, B = _setup("small", 5, cuda_device, use_tensor_cores=use_tc, power_law=1.5)
    deg = torch.bincount(d.edge_index[0], minlength=d.num_nodes)
    assert int(deg.max()) > 1000 and int((deg == 0).sum()) > 0
    _check_step(st, eng, train_idx[:B], cuda_device, apply_optim=False)


@pytest.mark.parametrize("name,seed", [("tiny", 0), ("small", 1), ("small", 2), ("cora", 0)])
def test_tensor_core_engine_step_parity(cuda_device, name, seed):
    """The same whole-step parity with the tcgen05 3xTF32 kernels in the loop: integer outputs and sampled sets stay
    bit-exact, logits / losses hold the 1e-5 bar, gradients hold it up to relu-kink flips (see _grad_ok)."""
    d, st, eng, train_idx, B = _setup(name, seed, cuda_device, use_tensor_cores=True)
    assert eng.use_tc and eng.use_tc_bwd
    _check_step(st, eng, train_idx[:B], cuda_device, apply_optim=False)


def test_tensor_core_engine_matches_simt_engine(cuda_device):
    """Mid-size frontier (several 128-row tiles per CTA, several 32-row blocks per CTA in the backward)."""
    from grapes_b200.synth import SHAPES
    kw = dict(N=40_000, E_dir=1_200_000, F=100, C=10, n_train=10_000, batch_size=256, num_samples=64, sampling_hops=2)
    SHAPES["mid"] = kw
    try:
        d, st, e_tc, train_idx, B = _setup("mid", 3, cuda_device, use_tensor_cores=True)
        _, _, e_simt, _, _ = _setup("mid", 3, cuda_device, use_tensor_cores=False)
    finally:
        SHAPES.pop("mid")
    assert e_tc.use_tc_bwd and not e_simt.use_tc
    t = train_idx[:B].to(cuda_device)
    noise = [torch.randn(e_tc.cap_n, device=cuda_device).abs().log().neg() for _ in range(2)]    # any fixed noise
    r1 = e_tc.step(t, gumbel_noise=noise, apply_optim=False, record=True)
    r2 = e_simt.step(t, gumbel_noise=noise, apply_optim=False, record=True)
    e_tc.check_overflow(); e_simt.check_overflow()
    for a, b in zip(r1["hops"], r2["hops"]):
        assert a["n"] > 5000
        assert torch.equal(a["sampled"], b["sampled"]) and torch.equal(a["batch_nodes"], b["batch_nodes"])
        assert _rel(a["logits_all"], b["logits_all"].cpu()) < TOL
    for k in ("loss_c", "tot_log_prob", "log_z", "loss_gfn"):
        assert abs(r1["scalars"][k] - r2["scalars"][k]) <= 4 * TOL * abs(r2["scalars"][k])
    for net in ("gcn_gf", "gcn_z"):
        for name, g2 in r2["grads"][net].items():
            g1 = r1["grads"][net][name]
            num = (g1.double() - g2.double()).norm() / g2.double().norm()
            assert num < 1e-4, f"{net}.{name}: relative L2 difference {num:.2e}"


def test_three_steps_with_adam(cuda_device):
    """Weights after optimiser steps track the float64 oracle.  Adam's first updates are ~ lr * sign(g): an entry
    whose gradient is zero up to rounding can take the other sign in ANY fp32 evaluation (the reference's own fp32
    run differs from float64 the same way), which moves that weight by up to 2*lr per step.  So: every weight within
    the sign-flip bound, and all but a small fraction within 1e-4 of the tensor's scale (the exact Adam arithmetic
    is pinned separately by test_adam_kernel_matches_torch_adam)."""
    d, st, eng, train_idx, B = _setup("cora", 2, cuda_device)
    nsteps = 2
    for i in range(nsteps):
        _check_step(st, eng, train_idx[i * B:(i + 1) * B], cuda_device, apply_optim=True, post_optim=(i > 0))
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
            assert frac <= max(0.01, 3.0 * frac32), f"{key} {name}: {frac:.4f} of the weights off by > 1e-4 (reference fp32: {frac32:.4f})"


def test_adam_kernel_matches_torch_adam(cuda_device):
    """Same gradients in -> same weights out as torch.optim.Adam (main.py:117-118), 6 steps."""
    from grapes_b200._lib import lib, ptr
    from grapes_b200.utils import _any_ctx
    gen = torch.Generator().manual_seed(0)
    n = 10_007
    p0 = torch.randn(n, generator=gen)
    ref = torch.nn.Parameter(p0.clone())
    opt = torch.optim.Adam([ref], lr=3e-3)
    p = p0.clone().to(cuda_device)
    m, v = torch.zeros_like(p), torch.zeros_like(p)
    step = torch.zeros(1, device=cuda_device)
    ctx = _any_ctx(cuda_device).ctx
    for i in range(6):
        g = torch.randn(n, generator=gen) * (10.0 ** (i - 3))
        ref.grad = g.clone()
        opt.step()
        gd = g.to(cuda_device)
        lib().grapes_adam_step(ctx, ptr(p), ptr(gd), ptr(m), ptr(v), n, 3e-3, 0.9, 0.999, 1e-8, ptr(step), 1,
                               torch.cuda.current_stream().cuda_stream)
    torch.testing.assert_close(p.cpu(), ref.detach(), rtol=1e-6, atol=1e-7)
    assert step.item() == 6.0


def test_step_parity_reinforce(cuda_device):
    d, st, eng, train_idx, B = _setup("tiny", 3, cuda_device, reinforce_baseline=True)
    _check_step(st, eng, train_idx[:B], cuda_device, apply_optim=False)


def test_step_parity_random_sampling(cuda_device):
    d, st, eng, train_idx, B = _setup("tiny", 4, cuda_device, random_sampling=True)
    _check_step(st, eng, train_idx[:B], cuda_device, apply_optim=False)


def test_step_parity_no_indicators_and_reg(cuda_device):
    d, st, eng, train_idx, B = _setup("tiny", 5, cuda_device, use_indicators=False, reg_param=0.1)
    _check_step(st, eng, train_idx[:B], cuda_device, apply_optim=False)


def test_step_parity_multilabel(cuda_device):
    d, st, eng, train_idx, B = _setup("tiny", 6, cuda_device, multilabel=True)
    _check_step(st, eng, train_idx[:B], cuda_device, apply_optim=False)


def test_take_all_branch_in_step(cuda_device):
    """num_samples >= #neighbours: the sampler keeps everything and draws no noise (utils.py:31-33)."""
    d, st, eng, train_idx, B = _setup("tiny", 7, cuda_device, num_samples=10_000)
    _check_step(st, eng, train_idx[:B], cuda_device, apply_optim=False)


def test_graph_replay_matches_eager(cuda_device):
    """The captured CUDA graph replays the same kernels: bitwise-identical weights, gradients and losses.  The eager
    warm-up before the first capture restores the Philox state, so both engines draw the same noise."""
    d, st, eng, train_idx, B = _setup("cora", 0, cuda_device)
    d2, st2, eng2, _, _ = _setup("cora", 0, cuda_device)
    for i in range(2):
        t = train_idx[i * B:(i + 1) * B].to(cuda_device)
        eng.step(t, use_graph=False)
        eng2.step(t, use_graph=True)
        torch.cuda.synchronize()
        assert torch.equal(eng.scal, eng2.scal), f"step {i}: losses differ between eager and graph replay"
        assert torch.equal(eng.all_nodes, eng2.all_nodes)
    eng.check_overflow(); eng2.check_overflow()
    assert torch.equal(eng.rng_state, eng2.rng_state)
    assert torch.equal(eng.grads, eng2.grads)
    assert torch.equal(eng.params, eng2.params)
    assert torch.equal(eng.exp_avg_sq, eng2.exp_avg_sq)
    assert eng2.count("A") > B


def test_determinism_run_to_run(cuda_device):
    d, st, eng, train_idx, B = _setup("small", 1, cuda_device)
    d2, st2, eng2, _, _ = _setup("small", 1, cuda_device)
    for e in (eng, eng2):
        e.step(train_idx[:B].to(cuda_device))
    torch.cuda.synchronize()
    assert torch.equal(eng.params, eng2.params)
    assert torch.equal(eng.grads, eng2.grads)


def test_prefetch_matches_plain_steps(cuda_device):
    """Cross-step prefetch (step(..., next_targets=...): reset + hop-0 front end of the next batch enqueued next to the
    classifier tail on the second step state) must not change a single bit: same batches, same Philox stream, Adam on;
    eager and CUDA-graph replay, with a partial last batch."""
    from grapes_b200.engine import GrapesEngine
    from grapes_b200.graph import DeviceGraph
    from grapes_b200.synth import SHAPES
    dev = cuda_device
    cfg = SHAPES["small"]
    d = make_synth("small", seed=4)
    g = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=dev)
    idx = d.train_mask.nonzero().squeeze(1).to(dev)
    B = cfg["batch_size"]
    batches = [idx[i * B:(i + 1) * B].to(torch.int32).contiguous() for i in range(6)]
    batches.append(idx[6 * B:6 * B + B // 2].to(torch.int32).contiguous())          # a partial last batch
    outs = {}
    for mode in ("plain", "prefetch"):
        for use_graph in (False, True):
            eng = GrapesEngine(g, d.x.to(dev), d.y.to(dev), num_classes=d.num_classes, batch_size=B,
                               num_samples=cfg["num_samples"], sampling_hops=cfg["sampling_hops"], seed=11)
            scal, nodes = [], []
            for j, b in enumerate(batches):
                nxt = batches[j + 1] if (mode == "prefetch" and j + 1 < len(batches)) else None
                eng.step(b, use_graph=use_graph, next_targets=nxt)
                scal.append(eng.scal.clone())
                nodes.append(eng.all_nodes.clone())
            eng.check_overflow()
            torch.cuda.synchronize()
            outs[(mode, use_graph)] = (eng.params.clone(), torch.stack(scal), torch.stack(nodes))
    ref = outs[("plain", False)]
    assert torch.isfinite(ref[1]).all()
    for key, val in outs.items():
        assert torch.equal(val[2], ref[2]), f"{key}: sampled subgraphs differ"
        assert torch.equal(val[1], ref[1]), f"{key}: losses differ"
        assert torch.equal(val[0], ref[0]), f"{key}: parameters differ"


@pytest.mark.parametrize("name,seed,tc", [("tiny", 0, False), ("small", 1, True), ("mid16", 2, True)])
def test_step_parity_bf16_feature_table(cuda_device, name, seed, tc):
    """papers100M-shaped config (BASELINE.json configs[4]): the feature table is stored as bf16.  Rows are gathered as
    stored and widened in the aggregation, arithmetic stays fp32, so against the oracle fed the same bf16-rounded values
    the fp32 bars hold (far inside the 2e-2 bf16 tolerance of the north star); integer contracts bit-exact.
    'mid16' (F = 128, frontier >= 4096 rows) takes the TMA-staged bf16 kernel, the others the warp-per-row form."""
    from grapes_b200.synth import SHAPES
    if name == "mid16":
        SHAPES["mid16"] = dict(N=30_000, E_dir=600_000, F=128, C=9, n_train=8_000, batch_size=256, num_samples=64,
                               sampling_hops=2)
    try:
        d, st, eng, train_idx, B = _setup(name, seed, cuda_device, use_tensor_cores=tc, feature_bf16=True)
    finally:
        SHAPES.pop("mid16", None)
    assert eng.x_bf16
    _check_step(st, eng, train_idx[:B], cuda_device, apply_optim=False)


def test_node_capacity_overflow_is_flagged_and_memory_safe(cuda_device):
    """A caller-chosen cap_nodes smaller than the frontier: the step must raise GRAPES_OVF_NODES (in the overflow word and
    in the step's flag scalar) and stay inside every buffer -- checked under compute-sanitizer memcheck with GRAPES_SANITIZE=1."""
    import os
    import shutil
    import subprocess
    import sys
    from grapes_b200._lib import GrapesError
    d, st, eng, train_idx, B = _setup("small", 1, cuda_device, use_tensor_cores=True, cap_nodes=700)
    assert eng.cap_n == 700
    eng.step(train_idx[:B].to(cuda_device), apply_optim=True)
    torch.cuda.synchronize()
    assert int(eng.overflow.item()) & 4
    assert int(eng.scalars()["flags"]) & 4                      # the tail launch copies the bits next to the losses
    with pytest.raises(GrapesError, match="nodes>cap_n"):
        eng.check_overflow()
    tool = shutil.which("compute-sanitizer") or "/usr/local/cuda/bin/compute-sanitizer"
    # opt-in (GRAPES_SANITIZE=1): B200_PROFILING.md allows one sanitizer OR ncu run per GPU lease, and the round-end
    # driver profiles with ncu in the lease that runs this suite.  (Not run in round 2: the GPU budget went elsewhere.)
    if os.environ.get("GRAPES_SANITIZE", "0") != "1" or not os.path.isfile(tool):
        return
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ("import sys, torch; sys.path.insert(0, %r); sys.path.insert(0, %r + '/tests');"
            "import test_gpu_engine as E; dev = torch.device('cuda:0');"
            "d, st, eng, tr, B = E._setup('small', 1, dev, use_tensor_cores=False, cap_nodes=700, multi_stream=False);"
            "eng.step(tr[:B].to(dev), apply_optim=True); torch.cuda.synchronize();"
            "assert int(eng.overflow.item()) & 4; print('SANITIZED')") % (root, root)
    res = subprocess.run([tool, "--error-exitcode", "9", "--launch-timeout", "0", sys.executable, "-c", code],
                         capture_output=True, text=True, timeout=900)
    assert res.returncode == 0 and "SANITIZED" in res.stdout, res.stdout[-3000:] + res.stderr[-2000:]
