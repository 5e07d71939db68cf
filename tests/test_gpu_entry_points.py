"""Entry points of include/grapes_b200.h that the engine calls on every step or on request, each through the C ABI
against an exact or float64 reference: the one-GPU step tail (grapes_step_tail without peers), the dropout-mask read-back
(grapes_dropout_mask), the forced scatter forms of the CSR builder, and the small list / bitmap / fill utilities.

Every output buffer starts as NaN (floats) or a sentinel (integers, bytes), so a write outside an entry point's contract
shows up as a changed sentinel."""
import ctypes

import numpy as np
import pytest
import torch

from dropout_utils import keep_mask, philox4x32_10
from oracle import reference_port as rp

pytestmark = pytest.mark.gpu

NAN = float("nan")
SENT = -7                                   # int32 sentinel
SENT_U8 = 0xAB


def _L():
    from grapes_b200._lib import lib
    return lib()


def _st():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    """device address of `t`; the caller keeps `t` alive until the launch is enqueued (a temporary freed earlier can be
    handed to the next allocation of the same call and overwritten before the kernel runs)"""
    return None if t is None else t.data_ptr()


def _i32(v, dev):
    return torch.tensor([v], dtype=torch.int32, device=dev)


def _bits(t):
    """the float32 tensor's bit patterns (NaN compares equal to the same NaN)"""
    return t.contiguous().view(torch.int32).cpu()


@pytest.fixture(scope="module")
def ctx(cuda_device):
    L = _L()
    c = ctypes.c_void_p()
    rc = L.cdll.grapes_ctx_create(cuda_device.index or 0, 1 << 16, 1 << 22, 1 << 20, ctypes.byref(c))
    assert rc == 0, L.last_error()
    yield c
    torch.cuda.synchronize()
    L.cdll.grapes_ctx_destroy(c)


# ---------------------------------------------------------------------------------------------------------------------
# grapes_step_tail without peers: the only optimiser launch of a one-GPU training step
# ---------------------------------------------------------------------------------------------------------------------
# (n, off0, n0, off1, n1, gf_off, n_gf, z_off, n_z): as the engine lays them out, the gcn_gf and gcn_z ranges sit inside
# group 1 (optimizer_gf); entries past both groups belong to no group
TAIL_LAYOUTS = {
    "many_blocks": (2**20 + 3, 0, 600_001, 600_001, 420_000, 600_001, 300_000, 900_001, 120_000),
    "empty_group0": (5000, 0, 0, 1000, 3000, 1000, 2000, 3000, 1000),
    # group 1 empty: the scaled ranges lie outside every group, so their gradients are written and nothing moves
    "empty_group1": (5000, 0, 2500, 2500, 0, 2500, 1500, 4000, 600),
}
LR0, LR1, B1, B2, EPS = 1e-3, 1e-4, 0.9, 0.999, 1e-8
COEF, LOG_Z_INIT = 0.5, 0.1


def _tail_inputs(n, dev, gen):
    p = torch.randn(n, generator=gen)
    m = torch.randn(n, generator=gen) * 1e-2
    v = torch.rand(n, generator=gen) * 1e-4
    d = torch.randn(n, generator=gen)
    return [t.to(dev) for t in (p, m, v, d)]


def _grads(n, gen, dev):
    g = torch.randn(n, generator=gen) * torch.pow(10.0, torch.rand(n, generator=gen) * 7 - 6)
    g[torch.rand(n, generator=gen) < 0.05] = 0.0
    return g.to(dev)


def _scal(dev):
    s = torch.full((16,), NAN, device=dev)
    s[0], s[1], s[2] = 1.3, -2.7, 0.4                     # loss_c, sum of log-probs, mean of the gcn_z logits
    return s


def _fp64_tail(p, m, v, g, d, steps, layout, do_scale, reinforce, have_log_z, scal):
    """float64 restatement: loss_gfn's gradient scale of the sampler ranges, then torch.optim.Adam on both groups (with the
    float32 values of the constants the launch receives)"""
    f = lambda x: float(np.float32(x))                    # noqa: E731
    n, off0, n0, off1, n1, gf_off, n_gf, z_off, n_z = layout
    p, m, v, g, d = (t.double().cpu() for t in (p, m, v, g, d))
    lc, tot, lzm = (float(x) for x in scal[:3].cpu())
    if do_scale:
        log_z = lzm - f(LOG_Z_INIT) if have_log_z else 0.0
        if reinforce:
            g_gf, g_z = -lc, 0.0
        else:
            r = log_z + tot + f(COEF) * lc
            g_gf = g_z = 2.0 * r
        g[gf_off:gf_off + n_gf] = g_gf * d[gf_off:gf_off + n_gf]
        g[z_off:z_off + n_z] = g_z * d[z_off:z_off + n_z]
    b1, b2 = f(B1), f(B2)
    for q, (o, k, lr) in enumerate(((off0, n0, f(LR0)), (off1, n1, f(LR1)))):
        t = float(steps[q]) + 1.0
        s = slice(o, o + k)
        m[s] = b1 * m[s] + (1 - b1) * g[s]
        v[s] = b2 * v[s] + (1 - b2) * g[s] ** 2
        p[s] = p[s] - lr / (1 - b1 ** t) * m[s] / (v[s].sqrt() / (1 - b2 ** t) ** 0.5 + f(EPS))
    return p, m, v, g


def _close_to_scale(got, ref, what):
    """within 1e-6 relative, or 1e-6 of the largest reference entry (a moment can cancel to almost nothing)"""
    torch.testing.assert_close(got.cpu().double(), ref, rtol=1e-6, atol=1e-6 * ref.abs().max().item(), msg=what)


@pytest.mark.parametrize("layout", list(TAIL_LAYOUTS))
@pytest.mark.parametrize("do_scale,reinforce,have_log_z", [(s, r, z) for s in (0, 1) for r in (0, 1) for z in (0, 1)])
def test_step_tail_without_peers(cuda_device, ctx, layout, do_scale, reinforce, have_log_z):
    """grapes_step_tail (peer_bufs NULL, world 1) == grapes_gfn_finalize_scale + grapes_adam_step2 bit for bit (it restates
    their arithmetic) over two calls in a row, and the first call against float64 at the tolerance of
    test_adam_step2_matches_torch_adam.  err_flag = 5 reaches scal[15]; step counts move only for non-empty groups; the
    state words (the last-block ticket) are back to zero after every call."""
    from grapes_b200._lib import lib
    L, dev = lib(), cuda_device
    lay = TAIL_LAYOUTS[layout]
    n, off0, n0, off1, n1, gf_off, n_gf, z_off, n_z = lay
    if not do_scale:
        n_gf = n_z = 0                                   # what the engine passes without a gradient scale
    gen = torch.Generator().manual_seed(n + 2 * do_scale + 4 * reinforce + 8 * have_log_z)
    p, m, v, d = _tail_inputs(n, dev, gen)
    A = dict(p=p.clone(), m=m.clone(), v=v.clone(), steps=torch.tensor([3.0, 7.0], device=dev), scal=_scal(dev))
    B = {k: t.clone() for k, t in A.items()}
    state = torch.zeros(int(L.cdll.grapes_peer_state_words()), dtype=torch.int32, device=dev)
    err = _i32(5, dev)
    f4 = 4                                               # bytes per float
    for call in range(2):
        g = _grads(n, gen, dev)
        A["g"], B["g"] = g.clone(), g.clone()
        if call == 0:
            first = (A["p"].clone(), A["m"].clone(), A["v"].clone(), g.clone(), A["steps"].clone())
        L.grapes_step_tail(ctx, _p(A["scal"]), do_scale, COEF, LOG_Z_INIT, reinforce, have_log_z, _p(d), gf_off, n_gf,
                           z_off, n_z, None, 0, 1, n, _p(A["p"]), _p(A["g"]), _p(A["m"]), _p(A["v"]), off0, n0, LR0, off1,
                           n1, LR1, B1, B2, EPS, _p(A["steps"]), _p(state), _p(err), _st())
        if do_scale:
            L.grapes_gfn_finalize_scale(ctx, _p(B["scal"]), COEF, LOG_Z_INIT, reinforce, have_log_z, _p(d) + f4 * gf_off,
                                        n_gf, _p(B["g"]) + f4 * gf_off, _p(d) + f4 * z_off, n_z, _p(B["g"]) + f4 * z_off,
                                        _st())
        L.grapes_adam_step2(ctx, _p(B["p"]), _p(B["g"]), _p(B["m"]), _p(B["v"]), off0, n0, LR0, off1, n1, LR1, B1, B2, EPS,
                            _p(B["steps"]), _st())
        torch.cuda.synchronize()
        for k in ("p", "m", "v", "g"):
            assert torch.equal(_bits(A[k]), _bits(B[k])), f"call {call}: {k} differs from finalize_scale + adam_step2"
        assert torch.equal(_bits(A["scal"][:15]), _bits(B["scal"][:15])), f"call {call}: scal"
        assert A["scal"][15].item() == 5.0, "err_flag does not reach scal[GRAPES_SCAL_FLAGS]"
        want = [3.0 + (call + 1) * (n0 > 0), 7.0 + (call + 1) * (n1 > 0)]
        assert A["steps"].tolist() == want == B["steps"].tolist(), f"call {call}: steps {A['steps'].tolist()}"
        assert not bool(state.any()), f"call {call}: state words not reset: {state.tolist()}"
        if call == 0:
            p64, m64, v64, g64 = _fp64_tail(*first[:4], d, first[4].tolist(), (n, off0, n0, off1, n1, gf_off, n_gf, z_off,
                                                                               n_z), do_scale, reinforce, have_log_z,
                                            A["scal"])
            torch.testing.assert_close(A["p"].cpu().double(), p64, rtol=1e-6, atol=1e-7)
            for k, ref in (("g", g64), ("m", m64), ("v", v64)):
                _close_to_scale(A[k], ref, k)
            live = torch.zeros(n, dtype=torch.bool)
            live[off0:off0 + n0] = True
            live[off1:off1 + n1] = True
            assert torch.equal(_bits(A["p"])[~live], _bits(first[0])[~live]), "a parameter outside both groups moved"
            assert torch.equal(_bits(A["m"])[~live], _bits(first[1])[~live])
            assert torch.equal(_bits(A["v"])[~live], _bits(first[2])[~live])


# ---------------------------------------------------------------------------------------------------------------------
# grapes_dropout_mask: the keep bits of a dropout site, read back for inspection and replay
# ---------------------------------------------------------------------------------------------------------------------
SEED = (0x5EED << 32) | 0x1234567               # both words of seed and step non-zero
STEP = (3 << 32) | 11


@pytest.mark.parametrize("rows,cap_rows,width", [(1, 1, 1), (97, 128, 3), (300, 300, 7), (1000, 1024, 13),
                                                 (513, 600, 256), (2049, 2049, 257), (0, 64, 5), (800, 700, 9)])
@pytest.mark.parametrize("thr", [0, 1 << 23, 1 << 24, 12_582_912])
def test_dropout_mask_matches_numpy(cuda_device, ctx, rows, cap_rows, width, thr):
    """keep[:min(rows, cap_rows) * width] == dropout_utils.keep_mask exactly; every byte past it keeps its sentinel"""
    dev = cuda_device
    tag = 3
    keep = torch.full((cap_rows * width + 64,), SENT_U8, dtype=torch.uint8, device=dev)
    rows_d = _i32(rows, dev)
    _L().grapes_dropout_mask(ctx, SEED, STEP, tag, thr, _p(rows_d), cap_rows, width, _p(keep), _st())
    torch.cuda.synchronize()
    r = min(rows, cap_rows)
    want = keep_mask(SEED, STEP, tag, thr, r, width).reshape(-1).astype(np.uint8)
    got = keep.cpu().numpy()
    assert np.array_equal(got[:r * width], want)
    assert (got[r * width:] == SENT_U8).all(), "a byte past rows * width was written"
    if thr == 0:
        assert not want.any()
    if thr == 1 << 24:
        assert want.all()


def _keep_at(idx, thr, tag):
    """keep bits of the entries idx (uint64 array) from Philox4x32-10 on the counters (i / 4, tag, step)"""
    words = philox4x32_10((idx >> np.uint64(2), tag, STEP & 0xFFFFFFFF, STEP >> 32), (SEED & 0xFFFFFFFF, SEED >> 32))
    w = np.stack(words, axis=1)[np.arange(idx.size), (idx & np.uint64(3)).astype(np.int64)]
    return ((w & np.uint64(0xFFFFFF)) < np.uint64(thr)).astype(np.uint8)


def test_dropout_mask_past_2_32_entries(cuda_device, ctx):
    """4.3 G entries (past 2^31 and 2^32): spot checks around both, at the start and at the end, and the sentinel past
    the device count"""
    dev = cuda_device
    rows, cap_rows, width, thr, tag = 4_300_000, 4_300_010, 1001, 1 << 23, 5
    total = rows * width
    assert total > 1 << 32
    keep = torch.full((cap_rows * width,), SENT_U8, dtype=torch.uint8, device=dev)
    rows_d = _i32(rows, dev)
    _L().grapes_dropout_mask(ctx, SEED, STEP, tag, thr, _p(rows_d), cap_rows, width, _p(keep), _st())
    torch.cuda.synchronize()
    idx = np.concatenate([np.arange(0, 4096), np.arange((1 << 31) - 2048, (1 << 31) + 2048),
                          np.arange((1 << 32) - 2048, (1 << 32) + 2048), np.arange(total - 4096, total)]).astype(np.uint64)
    got = keep[torch.from_numpy(idx.astype(np.int64)).to(dev)].cpu().numpy()
    assert np.array_equal(got, _keep_at(idx, thr, tag))
    assert bool((keep[total:] == SENT_U8).all()), "a byte past rows * width was written"
    del keep
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------------------------------
# grapes_csr_set_direct_scatter: the builder's forced grouping forms against scipy
# ---------------------------------------------------------------------------------------------------------------------
def _csr_cases():
    g = torch.Generator().manual_seed(0)
    for N, E in [(1, 5), (7, 40), (1000, 20000), (50000, 400000), (300, 90000)]:
        ei = torch.randint(0, N, (2, E), generator=g)                  # duplicates and self-loops at random
        yield f"multigraph_{N}", torch.cat([ei, ei[:, : E // 3], torch.arange(N).repeat(2, 1)[:, ::2]], dim=1), N
    for hub_deg in (33, 256, 257, 2048, 2049, 32768, 40000):           # a hub row in every per-row sort tier
        N = 60000
        cols = torch.randint(0, N, (hub_deg,), generator=g)
        cols[: hub_deg // 4] = cols[hub_deg // 4: 2 * (hub_deg // 4)]
        hub = torch.stack([torch.full((hub_deg,), 5), cols])
        rest = torch.randint(0, N, (2, 100000), generator=g)
        ei = torch.cat([hub, rest, hub.flip(0)], dim=1)[:, torch.randperm(2 * hub_deg + 100000, generator=g)]
        yield f"hub_{hub_deg}", ei, N
    yield "empty", torch.zeros((2, 0), dtype=torch.int64), 5
    yield "isolated", torch.tensor([[3], [3]]), 9
    yield "isolated_pair", torch.tensor([[0, 8, 8, 0], [8, 0, 0, 8]]), 9


@pytest.mark.parametrize("mode", [1, 2])
def test_csr_forced_scatter_forms_match_scipy(cuda_device, mode):
    """grapes_csr_set_direct_scatter(1) (one random scatter) and (2) (bucket partition + L2-windowed scatter) give scipy's
    canonical CSR on multigraphs, hub rows in every sort tier, the empty edge list and isolated nodes"""
    from grapes_b200.graph import csr_from_edge_index
    L = _L()
    try:
        L.grapes_csr_set_direct_scatter(mode)
        for name, ei, N in _csr_cases():
            adj = rp.build_adjacency(ei, N)
            indptr, indices = csr_from_edge_index(ei, N, cuda_device)
            assert np.array_equal(indptr.cpu().numpy(), adj.indptr.astype(np.int64)), name
            assert np.array_equal(indices.cpu().numpy(), adj.indices.astype(np.int32)), name
    finally:
        L.grapes_csr_set_direct_scatter(0)


# ---------------------------------------------------------------------------------------------------------------------
# list and bitmap utilities
# ---------------------------------------------------------------------------------------------------------------------
NODES = 10_000
WORDS = (NODES + 31) // 32


def _bitmap_of(ids, base=None):
    bm = np.zeros(WORDS, dtype=np.uint32) if base is None else base.copy()
    ids = np.asarray(ids, dtype=np.int64)
    np.bitwise_or.at(bm, ids >> 5, (np.uint32(1) << (ids & 31).astype(np.uint32)))
    return bm


def _u32(t):
    return t.cpu().numpy().view(np.uint32)


def _random_bitmap(gen, dev):
    bm = torch.randint(-2**31, 2**31 - 1, (WORDS,), generator=gen, dtype=torch.int64).to(torch.int32)
    bm[torch.rand(WORDS, generator=gen) < 0.7] = 0
    return bm.to(dev)


# (cap, count): full, one short, empty, clamped at the capacity; capacities off multiples of 32 and of 256
LIST_CASES = [(1000, 1000), (1000, 999), (257, 0), (300, 5000), (33, 17), (4099, 4001)]


@pytest.mark.parametrize("cap,count", LIST_CASES)
@pytest.mark.parametrize("with_b", [True, False])
def test_step_reset(cuda_device, ctx, cap, count, with_b):
    """targets -> the head of every row list, their bits ORed into bm_a (and bm_b), *P0 = min(count, cap)"""
    dev = cuda_device
    gen = torch.Generator().manual_seed(cap + count)
    targets = torch.randperm(NODES, generator=gen)[:cap].to(torch.int32)
    targets[cap // 2:] = targets[: cap - cap // 2].clone()           # repeated ids set the same bit twice
    targets_d, count_d = targets.to(dev), _i32(count, dev)
    nlists, stride = 4, cap + 13
    lists = torch.full((nlists * stride,), SENT, dtype=torch.int32, device=dev)
    bm_a, bm_b = _random_bitmap(gen, dev), _random_bitmap(gen, dev)
    a0, b0 = _u32(bm_a), _u32(bm_b)
    P0 = _i32(SENT, dev)
    _L().grapes_step_reset(ctx, _p(targets_d), _p(count_d), cap, _p(lists), stride, nlists, _p(P0),
                           _p(bm_a), _p(bm_b) if with_b else None, _st())
    torch.cuda.synchronize()
    n = min(count, cap)
    want = torch.full((nlists, stride), SENT, dtype=torch.int32)
    want[:, :n] = targets[:n]
    assert torch.equal(lists.cpu().view(nlists, stride), want)
    assert int(P0) == n
    assert np.array_equal(_u32(bm_a), _bitmap_of(targets[:n].numpy(), a0))
    assert np.array_equal(_u32(bm_b), _bitmap_of(targets[:n].numpy(), b0) if with_b else b0)


@pytest.mark.parametrize("cap,count", LIST_CASES)
@pytest.mark.parametrize("off", [0, 33])
@pytest.mark.parametrize("with_total", [True, False])
def test_append_list(cuda_device, ctx, cap, count, off, with_total):
    """dst[off .. off + n) = src[:n], n = min(count, cap); *total = off + n; nothing else written"""
    dev = cuda_device
    src = torch.randint(0, NODES, (cap,), generator=torch.Generator().manual_seed(cap), dtype=torch.int32)
    dst = torch.full((off + cap + 50,), SENT, dtype=torch.int32, device=dev)
    total = _i32(SENT, dev)
    src_d, count_d = src.to(dev), _i32(count, dev)
    _L().grapes_append_list(ctx, _p(src_d), _p(count_d), cap, _p(dst), off,
                            _p(total) if with_total else None, _st())
    torch.cuda.synchronize()
    n = min(count, cap)
    want = torch.full((off + cap + 50,), SENT, dtype=torch.int32)
    want[off:off + n] = src[:n]
    assert torch.equal(dst.cpu(), want)
    assert int(total) == (off + n if with_total else SENT)


@pytest.mark.parametrize("n", [0, 1, 255, 256, 257, 100_003])
@pytest.mark.parametrize("with_count", [True, False])
def test_ids_i64_to_i32(cuda_device, ctx, n, with_count):
    """out[:n] = int32(in[:n]) over the whole int32 range; *count = n; nothing past n written"""
    dev = cuda_device
    src = torch.randint(-2**31, 2**31, (n,), generator=torch.Generator().manual_seed(n), dtype=torch.int64)
    src[: min(n, 3)] = torch.tensor([-2**31, 2**31 - 1, -1])[: min(n, 3)]
    out = torch.full((n + 40,), SENT, dtype=torch.int32, device=dev)
    cnt = _i32(SENT, dev)
    src_d = src.to(dev) if n else None
    _L().grapes_ids_i64_to_i32(ctx, _p(src_d), n, _p(out), _p(cnt) if with_count else None, _st())
    torch.cuda.synchronize()
    assert torch.equal(out.cpu()[:n], src.to(torch.int32))
    assert bool((out.cpu()[n:] == SENT).all())
    assert int(cnt) == (n if with_count else SENT)


@pytest.mark.parametrize("cap,count", LIST_CASES + [(0, 0)])
@pytest.mark.parametrize("with_count", [True, False])
def test_ids_i32_to_i64(cuda_device, ctx, cap, count, with_count):
    """out[:n] = int64(in[:n]), n = min(count, cap) (cap without a count); nothing past n written"""
    dev = cuda_device
    src = torch.randint(-2**31, 2**31, (cap,), generator=torch.Generator().manual_seed(cap), dtype=torch.int64)
    src = src.to(torch.int32)
    out = torch.full((cap + 40,), SENT, dtype=torch.int64, device=dev)
    src_d = src.to(dev) if cap else None
    count_d = _i32(count, dev)
    _L().grapes_ids_i32_to_i64(ctx, _p(src_d), _p(count_d) if with_count else None, cap, _p(out), _st())
    torch.cuda.synchronize()
    n = min(count, cap) if with_count else cap
    assert torch.equal(out.cpu()[:n], src[:n].to(torch.int64))
    assert bool((out.cpu()[n:] == SENT).all())


@pytest.mark.parametrize("cap,count", LIST_CASES)
def test_bitmap_set_and_clear_words(cuda_device, ctx, cap, count):
    """grapes_bitmap_set ORs the bits of ids[:n] into a bitmap that already holds others; grapes_bitmap_clear_words
    zeroes every word that holds one of ids2[:n], n = min(count, cap), and no other word"""
    dev = cuda_device
    gen = torch.Generator().manual_seed(3 * cap + count)
    ids = torch.randint(0, NODES, (cap,), generator=gen, dtype=torch.int32)
    ids2 = torch.randint(0, NODES, (cap,), generator=gen, dtype=torch.int32)
    bm = _random_bitmap(gen, dev)
    b0 = _u32(bm)
    n = min(count, cap)
    L = _L()
    ids_d, ids2_d, count_d = ids.to(dev), ids2.to(dev), _i32(count, dev)
    L.grapes_bitmap_set(ctx, _p(ids_d), _p(count_d), cap, _p(bm), _st())
    torch.cuda.synchronize()
    want = _bitmap_of(ids[:n].numpy(), b0)
    assert np.array_equal(_u32(bm), want)
    L.grapes_bitmap_clear_words(ctx, _p(ids2_d), _p(count_d), cap, _p(bm), _st())
    torch.cuda.synchronize()
    want[ids2[:n].numpy() >> 5] = 0
    assert np.array_equal(_u32(bm), want)


SIZES = [0, 1, 255, 256, 257, 100_003, 2**20 + 3]


@pytest.mark.parametrize("n", SIZES)
def test_scale_by_device_scalar(cuda_device, ctx, n):
    """grad[:n] = (*g) * dir[:n] in float32 (bit for bit the torch product); nothing past n written"""
    dev = cuda_device
    d = torch.randn(max(n, 1), generator=torch.Generator().manual_seed(n))      # n = 0: a valid pointer, nothing read
    g = torch.tensor([-1.7], dtype=torch.float32)
    grad = torch.full((n + 37,), NAN, device=dev)
    d_d, g_d = d.to(dev), g.to(dev)
    _L().grapes_scale_by_device_scalar(ctx, _p(d_d), _p(g_d), n, _p(grad), _st())
    torch.cuda.synchronize()
    assert torch.equal(_bits(grad[:n]), _bits(g * d[:n]))
    assert bool(torch.isnan(grad[n:]).all())


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("value", [3.25, -0.0])
def test_fill_f32(cuda_device, ctx, n, value):
    dev = cuda_device
    p = torch.full((n + 37,), NAN, device=dev)
    _L().grapes_fill_f32(ctx, _p(p), value, n, _st())
    torch.cuda.synchronize()
    assert torch.equal(_bits(p[:n]), _bits(torch.full((n,), value)))
    assert bool(torch.isnan(p[n:]).all())


@pytest.mark.parametrize("nbytes", [0, 1, 13, 4096, 100_003])
def test_zero(cuda_device, ctx, nbytes):
    """exactly `nbytes` bytes from an address off 16-byte alignment; NULL with 0 bytes is accepted"""
    dev = cuda_device
    buf = torch.full((nbytes + 64,), SENT_U8, dtype=torch.uint8, device=dev)
    L = _L()
    L.grapes_zero(ctx, buf.data_ptr() + 3, nbytes, _st())
    L.grapes_zero(ctx, None, 0, _st())
    torch.cuda.synchronize()
    got = buf.cpu()
    assert bool((got[3:3 + nbytes] == 0).all())
    assert bool((got[:3] == SENT_U8).all()) and bool((got[3 + nbytes:] == SENT_U8).all())
