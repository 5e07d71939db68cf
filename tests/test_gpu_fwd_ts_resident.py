"""grapes_sampler_l1_fwd_tc -- the sampler head's tensor-core forward, z = relu(Y W1^T + b1) . w2 with its relu mask bits --
with W resident in shared memory and every CTA walking many row tiles, row by row against float64, through the C ABI.

With Y_lo = None the call runs k_l1_fwd_ts, which keeps the CTA's 128-column half of W resident for K <= 160 (at most 5
k-blocks of 32); with the presplit (Y_hi, Y_lo) pair it runs k_l1_fwd_tc, resident for K <= 128.  A resident CTA owns one
column half and walks the row tiles t = first, first + per_half, ... (per_half = SMs / (D / 128)), while the raw Y tiles
pass through a ring of at most 8 shared-memory slots that the TMA refills as soon as the converter warps release one.  Every
case sizes n so that each CTA walks WALK tiles, more than the ring holds, so every slot is refilled many times while the
converters still work on the tile before.  That is the regime in which the converters of k_l1_fwd_ts used to release a slot
before their reads of it had been performed: the dense-layer instantiation of the kernel then read chunks of the slot's next
fill (tests/test_gpu_dense_tc.py holds that instantiation in the same regime).

Per row r, against float64: |z_r - ref_r| <= 1e-5 * sum_d |relu(pre_rd) w2_d| (+ 1e-6), the row's own scale and not a
global maximum; maskT bits equal pre > 0 wherever |pre| clears the relu kink.  zpart starts as NaN and maskT as all ones:
zpart columns at or past n and the maskT row groups past the last tile must keep them.  Y holds NaN in its rows past n and
its pitch columns past K.  Two launches give the same bits, and so does the same call with W streamed (grapes_tc_debug
bit 1): both forms add in the same order."""
import ctypes

import pytest
import torch

pytestmark = pytest.mark.gpu

NAN = float("nan")
TOL = 1e-5
TINY = 1e-6
KINK = 1e-4                     # |pre| above this is clear of the relu kink (inputs of unit scale)
WALK = 10                       # row tiles per CTA: more than the deepest Y ring (8 slots) + 2
D_ALL = (128, 256, 384, 512)
K_ALL = (15, 32, 33, 100, 104, 131, 160, 161)     # 1 to 5 k-blocks, each count entered and left; 161: W streamed


def _L():
    from grapes_b200._lib import lib
    return lib()


def _st():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


def _new_ctx(dev, sm_limit=0):
    L = _L()
    c = ctypes.c_void_p()
    rc = L.cdll.grapes_ctx_create(dev.index or 0, 1, 1 << 20, 1 << 20, ctypes.byref(c))
    assert rc == 0, L.last_error()
    if sm_limit:
        L.grapes_ctx_set_sm_limit(c, sm_limit)
    return c


@pytest.fixture(scope="module")
def ctxs(cuda_device):
    """{"full": every SM, "one": limited to one SM}"""
    out = {"full": _new_ctx(cuda_device), "one": _new_ctx(cuda_device, sm_limit=1)}
    yield out
    torch.cuda.synchronize()
    for c in out.values():
        _L().cdll.grapes_ctx_destroy(c)


def _walk_rows(dev, D):
    """n at which every CTA of each column half walks WALK row tiles and one CTA a partial tile more"""
    per_half = torch.cuda.get_device_properties(dev).multi_processor_count // (D // 128)
    return WALK * per_half * 128 + 77


class _Case:
    """Y [cap_n, ldy] with N(0, 1) in rows < n and columns < K, NaN elsewhere; Glorot W1; b1, w2 ~ 0.1 N(0, 1); the 3xTF32
    split of W1 and, for presplit, of all ldy columns of Y (so the pair carries the NaN guards too)"""

    def __init__(self, ctx, dev, n, K, D, presplit, seed):
        g = torch.Generator(device=dev).manual_seed(seed)
        self.ctx, self.n, self.K, self.D = ctx, n, K, D
        self.cap_n = n + 300
        ldy = (K + 3) // 4 * 4 + 4
        self.Y = torch.full((self.cap_n, ldy), NAN, device=dev)
        self.Y[:n, :K] = torch.randn(n, K, generator=g, device=dev)
        self.W = (torch.rand(D, K, generator=g, device=dev) * 2 - 1) * (6.0 / (D + K)) ** 0.5
        self.b1 = torch.randn(D, generator=g, device=dev) * 0.1
        self.w2 = torch.randn(D, generator=g, device=dev) * 0.1
        self.ldw = (K + 3) // 4 * 4
        self.Wh, self.Wl = (torch.empty((D, self.ldw), device=dev) for _ in range(2))
        L = _L()
        L.grapes_split_tf32(ctx, _p(self.W), K, D, K, _p(self.Wh), _p(self.Wl), self.ldw, _st())
        self.Ya, self.Yb = self.Y, None
        if presplit:
            self.Ya, self.Yb = torch.empty_like(self.Y), torch.empty_like(self.Y)
            L.grapes_split_tf32(ctx, _p(self.Y), ldy, self.cap_n, ldy, _p(self.Ya), _p(self.Yb), ldy, _st())

    def run(self, stream_w=False):
        """one launch into fresh sentinel-filled zpart / maskT; (zpart, maskT) once it has finished"""
        dev = self.Y.device
        zpart = torch.full((2 * (self.D // 128), self.cap_n), NAN, device=dev)
        maskT = torch.full(((self.cap_n + 127) // 128 * 4, self.D), -1, dtype=torch.int32, device=dev)
        cnt = torch.tensor([self.n], dtype=torch.int32, device=dev)
        L = _L()
        L.cdll.grapes_tc_debug(2 if stream_w else 0)
        try:
            L.grapes_sampler_l1_fwd_tc(self.ctx, _p(self.Ya), _p(self.Yb), self.Y.stride(0), _p(cnt), self.cap_n, self.K,
                                       _p(self.Wh), _p(self.Wl), self.ldw, self.D, _p(self.b1), _p(self.w2), _p(zpart),
                                       _p(maskT), _st())
            torch.cuda.synchronize()
        finally:
            L.cdll.grapes_tc_debug(0)
        return zpart, maskT

    def check(self, zpart, maskT, what):
        n, K = self.n, self.K
        pre = self.Y[:n, :K].double() @ self.W.double().t() + self.b1.double()
        terms = torch.relu(pre) * self.w2.double()
        ref, scale = terms.sum(1), terms.abs().sum(1)
        del terms
        z = zpart[:, :n].double().sum(0)
        bad = ~((z - ref).abs() <= TOL * scale + TINY)             # NaN counts as bad
        if bool(bad.any()):
            rows = bad.nonzero().squeeze(1)
            r = int(rows[0])
            pytest.fail(f"{what}: {rows.numel()} of {n} rows off their float64 value, first row {r} (tile {r // 128}): "
                        f"z {float(z[r]):.7g}, float64 {float(ref[r]):.7g}, row scale {float(scale[r]):.4g}")
        assert bool(torch.isnan(zpart[:, n:]).all()), f"{what}: a zpart column at or past n was written"
        m_tiles = (n + 127) // 128
        assert bool((maskT[m_tiles * 4:] == -1).all()), f"{what}: a maskT row group past the last row tile was written"
        rows = torch.arange(n, device=pre.device)
        bits = ((maskT[rows // 32] >> (rows % 32).unsqueeze(1)) & 1).bool()
        clear = pre.abs() > KINK
        wrong = (bits != (pre > 0)) & clear
        assert not bool(wrong.any()), f"{what}: {int(wrong.sum())} relu mask bits clear of the kink differ from float64"


def _run(ctx, dev, n, K, D, presplit, seed, what):
    c = _Case(ctx, dev, n, K, D, presplit, seed)
    z1, m1 = c.run()
    c.check(z1, m1, what)
    z2, m2 = c.run()
    assert torch.equal(z1.view(torch.int32), z2.view(torch.int32)), f"{what}: zpart differs between two launches"
    assert torch.equal(m1, m2), f"{what}: maskT differs between two launches"
    z3, m3 = c.run(stream_w=True)
    assert torch.equal(z1.view(torch.int32), z3.view(torch.int32)), f"{what}: zpart differs with W streamed"
    assert torch.equal(m1, m3), f"{what}: maskT differs with W streamed"


@pytest.mark.parametrize("presplit", [False, True], ids=["fwd_ts", "presplit_fwd_tc"])
@pytest.mark.parametrize("D", D_ALL)
@pytest.mark.parametrize("K", K_ALL)
def test_resident_walk_matches_fp64(cuda_device, ctxs, K, D, presplit):
    """every resident k-block count, the first streamed K and every hidden width, each CTA walking WALK row tiles"""
    n = _walk_rows(cuda_device, D)
    _run(ctxs["full"], cuda_device, n, K, D, presplit, seed=K * 1000 + D + presplit, what=f"n={n} K={K} D={D}")


@pytest.mark.parametrize("presplit", [False, True], ids=["fwd_ts", "presplit_fwd_tc"])
def test_resident_walk_past_150k_rows(cuda_device, ctxs, presplit):
    """the products-shaped head (K = 104, D = 256) over 160 007 rows: 16 to 17 row tiles per CTA"""
    _run(ctxs["full"], cuda_device, 160_007, 104, 256, presplit, seed=17, what="n=160007 K=104 D=256")


@pytest.mark.parametrize("presplit", [False, True], ids=["fwd_ts", "presplit_fwd_tc"])
@pytest.mark.parametrize("K", [15, 104, 128])
def test_resident_one_sm(cuda_device, ctxs, K, presplit):
    """a context limited to one SM at D = 128: one resident CTA walks all 391 row tiles"""
    _run(ctxs["one"], cuda_device, 50_000, K, 128, presplit, seed=K + 5, what=f"one SM, K={K}")
