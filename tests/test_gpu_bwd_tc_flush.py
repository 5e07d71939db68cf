"""grapes_sampler_l1_bwd_tc -- the sampler head's tensor-core backward, S = (dz * mask)^T [Y | 1] and from it
scale * d(sum_r dz_r z_r) / d(W1, b1, w2) added onto the gradients -- element by element against float64, through the
C ABI, in the regimes production runs and the older tests never reach.

With Y_lo = None the call runs k_l1_bwd_ts.  Its grid is (per_half * D/128, nchunks): a CTA owns one 128-unit half of the
hidden layer and one 128-column chunk of [Y | 1], and takes the row groups (32 rows) pp, pp + per_half, ... with
per_half = SMs / nchunks / (D/128).  The tensor core adds into its fp32 accumulator with truncation, so every CTA cuts its
accumulator chain every TCBS_FLUSH = 96 groups: each interval goes to a slab part[flush][pp][D][N] of its own, slabs past
the CTA's last interval (nflush is sized on the host from cap_n) are filled with zeros, and k_l1_bwd_finalize adds
per_half * nflush slabs and walks the chunks in order.  A Reddit-shaped hop (154 k rows, 606 columns) runs 4 intervals per
CTA.  grapes_tc_debug bit 8, or a presplit (Y_hi, Y_lo) pair, runs k_l1_bwd_tc instead: its CTAs cover both halves and
deal the row groups out over SMs / nchunks CTAs per chunk, with the same flush intervals, slabs and zero-fill.  (Before
it had them, one chain of 1563 same-sign groups drifted 1.9e-4 of the magnitude: test_same_sign_worst_case.)

The relu mask is built here, as maskT[(rows / 32)][D] words: bits of a float64 `pre > 0`, random bits, all ones or all
zeros, so the backward is tested on its own.  Per element, with m the mask bits and every factor replaced by its absolute
value for the magnitude (plus |g0|):  |got - ref| <= 1e-5 * mag + 1e-6.  Y rows in [n, cap_n) hold 1e30 (finite, as the
kernels require of the rows of the last group), dz[n:] is NaN and the mask bits of rows >= n are all ones: none of it may
reach the gradients.  The gradients start from nonzero g0 and the calls use scale 1.0 and -0.37, as the engine adds the
backward of every hop into the same buffers."""
import ctypes

import pytest
import torch

pytestmark = pytest.mark.gpu

NAN = float("nan")
TOL = 1e-5
TINY = 1e-6
FLUSH = 96                      # TCBS_FLUSH of k_l1_bwd_ts (groups of 32 rows per accumulator chain)
ROWS = 32
BIG = 1e30                      # Y rows past n: finite, so 0 * Y stays 0


def _L():
    from grapes_b200._lib import lib
    return lib()


def _st():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


def _new_ctx(dev, partials_bytes, sm_limit=0):
    L = _L()
    c = ctypes.c_void_p()
    rc = L.cdll.grapes_ctx_create(dev.index or 0, 1, 1 << 20, partials_bytes, ctypes.byref(c))
    assert rc == 0, L.last_error()
    if sm_limit:
        L.grapes_ctx_set_sm_limit(c, sm_limit)
    return c


@pytest.fixture(scope="module")
def ctxs(cuda_device):
    """{"full": every SM, "one": limited to one SM, "small": every SM with the smallest partial buffer (1 MB)}"""
    out = {"full": _new_ctx(cuda_device, 256 << 20), "one": _new_ctx(cuda_device, 256 << 20, sm_limit=1),
           "small": _new_ctx(cuda_device, 1 << 20)}
    yield out
    torch.cuda.synchronize()
    for c in out.values():
        _L().cdll.grapes_ctx_destroy(c)


def _sms(dev, which):
    return 1 if which == "one" else torch.cuda.get_device_properties(dev).multi_processor_count


def _ts_grid(sms, ncols, D, cap_n):
    """(per_half, nflush) as grapes_sampler_l1_bwd_tc sizes k_l1_bwd_ts"""
    nchunks, max_groups = -(-ncols // 128), -(-cap_n // ROWS)
    per_half = min(max(1, sms // nchunks // (D // 128)), max_groups)
    return per_half, -(-(-(-max_groups // per_half)) // FLUSH)


def _rows_for(per_half, g0_groups):
    """n at which CTA 0 of every half gets exactly g0_groups row groups (the others one less), the last one partial"""
    return ((g0_groups - 1) * per_half) * ROWS + 17


def _pack(bits):
    """bool [rows (multiple of 32), D] -> maskT int32 [rows / 32, D], bit i of word (g, d) = row 32 g + i"""
    G, D = bits.shape[0] // ROWS, bits.shape[1]
    sh = torch.arange(ROWS, device=bits.device, dtype=torch.int64).view(1, ROWS, 1)
    w = (bits.view(G, ROWS, D).to(torch.int64) << sh).sum(1)
    return torch.where(w >= 2 ** 31, w - 2 ** 32, w).to(torch.int32)


class _Case:
    """one backward problem: Y [cap_n, ldy] (features, `extra` indicator columns, the ones column, NaN pitch), dz, W1 with
    a NaN pitch column, b1, w2, the mask bits and nonzero starting gradients g0"""

    def __init__(self, dev, n, cap_n, K, extra, D, mask="pre", seed=0, same_sign=False):
        g = torch.Generator(device=dev).manual_seed(seed)
        self.dev, self.n, self.cap_n, self.K, self.D = dev, n, cap_n, K, D
        self.ones_col = K + extra
        self.ncols = self.ones_col + 1
        ldy = (self.ncols + 3) // 4 * 4 + 4
        rnd = (lambda *s: torch.rand(*s, generator=g, device=dev)) if same_sign else \
              (lambda *s: torch.randn(*s, generator=g, device=dev))
        self.Y = torch.full((cap_n, ldy), NAN, device=dev)
        self.Y[:n, :K] = rnd(n, K)
        self.Y[:n, K:self.ones_col] = (torch.rand(n, extra, generator=g, device=dev) < 0.3).float()   # indicators
        self.Y[:n, self.ones_col] = 1.0
        self.Y[n:, :self.ncols] = BIG
        self.dz = torch.full((cap_n,), NAN, device=dev)
        self.dz[:n] = (torch.rand(n, generator=g, device=dev) + 0.05) if same_sign else torch.randn(n, generator=g, device=dev)
        self.ldw = K + 1
        self.W1 = torch.full((D, self.ldw), NAN, device=dev)
        self.W1[:, :K] = (torch.rand(D, K, generator=g, device=dev) * 2 - 1) * (6.0 / (D + K)) ** 0.5
        self.b1 = torch.randn(D, generator=g, device=dev) * 0.1
        self.w2 = (torch.rand(D, generator=g, device=dev) * 0.1 + 0.01) if same_sign else \
            torch.randn(D, generator=g, device=dev) * 0.1
        rows = (cap_n + ROWS - 1) // ROWS * ROWS
        bits = torch.ones((rows, D), dtype=torch.bool, device=dev)          # rows >= n: all ones
        if mask == "pre":
            pre = self.Y[:n, :K].double() @ self.W1[:, :K].double().t() + self.b1.double()
            bits[:n] = pre > 0
            del pre
        elif mask == "random":
            bits[:n] = torch.rand(n, D, generator=g, device=dev) < 0.5
        elif mask == "zeros":
            bits[:n] = False
        else:
            assert mask == "ones"
        self.bits = bits[:n]
        self.maskT = _pack(bits)
        zero = same_sign
        self.g0 = tuple(torch.zeros(*s, device=dev) if zero else torch.randn(*s, generator=g, device=dev)
                        for s in ((D, K), (D,), (D,)))
        self.Yhi = self.Ylo = None
        self._ref = {}

    def presplit(self, ctx):
        if self.Yhi is None:
            ldy = self.Y.shape[1]
            self.Yhi, self.Ylo = torch.empty_like(self.Y), torch.empty_like(self.Y)
            _L().grapes_split_tf32(ctx, _p(self.Y), ldy, self.cap_n, ldy, _p(self.Yhi), _p(self.Ylo), ldy, _st())
        return self.Yhi, self.Ylo

    def args(self, ctx, n_dev, Ya, Yb, scale, grads):
        return (ctx, _p(Ya), _p(Yb), self.Y.shape[1], self.ncols, _p(n_dev), self.cap_n, self.K,
                self.ones_col, _p(self.maskT), _p(self.W1), self.ldw, self.D, _p(self.b1), _p(self.w2), _p(self.dz),
                scale, _p(grads[0]), _p(grads[1]), _p(grads[2]), _st())

    def run(self, ctx, kernel="ts", scale=1.0, n=None):
        """one call from fresh copies of g0; the gradients once it has finished.  kernel: "ts" (default), "tc"
        (grapes_tc_debug bit 8) or "presplit" (the (Y_hi, Y_lo) pair, k_l1_bwd_tc)"""
        grads = tuple(t.clone() for t in self.g0)
        n_dev = torch.tensor([self.n if n is None else n], dtype=torch.int32, device=self.dev)
        Ya, Yb = self.presplit(ctx) if kernel == "presplit" else (self.Y, None)
        L = _L()
        L.cdll.grapes_tc_debug(8 if kernel == "tc" else 0)
        try:
            L.grapes_sampler_l1_bwd_tc(*self.args(ctx, n_dev, Ya, Yb, scale, grads))
            torch.cuda.synchronize()
        finally:
            L.cdll.grapes_tc_debug(0)
        return grads

    def ref(self, n, scale):
        """float64 (gW1, gb1, gw2) and their magnitudes for the first n rows"""
        key = (n, scale)
        if key not in self._ref:
            K, oc = self.K, self.ones_col
            A = self.dz[:n].double().unsqueeze(1) * self.bits[:n].double()              # [n, D]
            Yx = self.Y[:n, :self.ncols].double()
            S, Sm = A.t() @ Yx, A.abs().t() @ Yx.abs()
            del A, Yx
            w2, b1, W1 = self.w2.double(), self.b1.double(), self.W1[:, :K].double()
            g0 = [t.double() for t in self.g0]
            sw = scale * w2
            ref = (g0[0] + sw.unsqueeze(1) * S[:, :K], g0[1] + sw * S[:, oc],
                   g0[2] + scale * ((W1 * S[:, :K]).sum(1) + b1 * S[:, oc]))
            mag = (g0[0].abs() + sw.abs().unsqueeze(1) * Sm[:, :K], g0[1].abs() + sw.abs() * Sm[:, oc],
                   g0[2].abs() + abs(scale) * ((W1.abs() * Sm[:, :K]).sum(1) + b1.abs() * Sm[:, oc]))
            self._ref[key] = (ref, mag)
        return self._ref[key]

    def worst(self, got, scale=1.0, n=None):
        """the largest |err| / mag over the three gradients"""
        ref, mag = self.ref(self.n if n is None else n, scale)
        return max(float(((gt.double() - rf).abs() / mg.clamp_min(1e-300)).max()) for gt, rf, mg in zip(got, ref, mag))

    def check(self, got, what, scale=1.0, n=None):
        """every element within its own bound"""
        ref, mag = self.ref(self.n if n is None else n, scale)
        for name, gt, rf, mg in zip(("gW1", "gb1", "gw2"), got, ref, mag):
            err = (gt.double() - rf).abs()
            bad = ~(err <= TOL * mg + TINY)                              # NaN counts as bad
            if bool(bad.any()):
                idx = bad.nonzero()[0].tolist()
                where = f"d {idx[0]}, k {idx[1]}, chunk {idx[1] // 128}" if name == "gW1" else \
                    f"d {idx[0]}, chunk {self.ones_col // 128}" if name == "gb1" else f"d {idx[0]}, all chunks"
                pytest.fail(f"{what}: {int(bad.sum())} of {bad.numel()} {name} elements off their float64 value, first "
                            f"({where}): got {float(gt[tuple(idx)]):.8g}, float64 {float(rf[tuple(idx)]):.8g}, "
                            f"magnitude {float(mg[tuple(idx)]):.4g}")


def _bits_equal(a, b):
    return all(torch.equal(x.view(torch.int32), y.view(torch.int32)) for x, y in zip(a, b))


def _check_ts(c, ctx, what, scale, tc=()):
    """k_l1_bwd_ts twice (identical bits) against float64; then each k_l1_bwd_tc form in `tc`"""
    g1 = c.run(ctx, "ts", scale)
    c.check(g1, f"{what} [bwd_ts]", scale)
    g2 = c.run(ctx, "ts", scale)
    assert _bits_equal(g1, g2), f"{what}: k_l1_bwd_ts differs between two launches"
    for kern in tc:
        c.check(c.run(ctx, kern, scale), f"{what} [{kern}]", scale)


# ---- flush boundaries ------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("which", ["full", "one"])
@pytest.mark.parametrize("D", [128, 256])
@pytest.mark.parametrize("groups0", [95, 96, 97, 192, 193])
def test_flush_boundaries(cuda_device, ctxs, which, D, groups0):
    """CTA 0 of each half walks exactly 95, 96, 97, 192 or 193 row groups (the others one less): the last group of an
    interval, the first of the next, and CTAs that end one interval short of CTA 0 and zero-fill the slab"""
    K, extra = 20, 3
    ncols = K + extra + 1
    P, _ = _ts_grid(_sms(cuda_device, which), ncols, D, 1 << 30)
    n = _rows_for(P, groups0)
    cap_n = n + 10                                                   # nflush = CTA 0's intervals
    per_half, nflush = _ts_grid(_sms(cuda_device, which), ncols, D, cap_n)
    assert per_half == P and nflush == -(-groups0 // FLUSH)
    c = _Case(cuda_device, n, cap_n, K, extra, D, mask="pre" if groups0 % 2 else "random", seed=groups0 * 7 + D)
    scale = -0.37 if groups0 % 2 else 1.0
    _check_ts(c, ctxs[which], f"{which} D={D} CTA 0 walks {groups0} groups (n={n})", scale,
              tc=("tc",) if which == "one" else ())           # one SM: k_l1_bwd_tc's one CTA walks the same groups


def test_idle_ctas(cuda_device, ctxs):
    """fewer row groups than CTAs per half: the last CTAs of each half get no group and only fill their slabs with zeros"""
    D, K = 256, 104
    per_half, _ = _ts_grid(_sms(cuda_device, "full"), K + 1, D, 1 << 30)
    n = (per_half // 3) * ROWS + 5
    c = _Case(cuda_device, n, per_half * ROWS * 2, K, 0, D, mask="random", seed=3)
    _check_ts(c, ctxs["full"], f"idle CTAs (n={n})", -0.37, tc=("tc", "presplit"))


# ---- column chunks ---------------------------------------------------------------------------------------------------

CHUNKS = [(15, 0), (30, 2), (127, 0), (125, 3), (602, 3), (1433, 3)]     # ncols 16, 33, 128, 129, 606, 1437


@pytest.mark.parametrize("K,extra", CHUNKS, ids=[f"ncols{K + e + 1}" for K, e in CHUNKS])
def test_column_chunks(cuda_device, ctxs, K, extra):
    """one to twelve 128-column chunks, indicator columns between K and the ones column, the ones column alone in the last
    chunk (ncols 129): on every SM, and on one SM where every CTA runs several flush intervals in every chunk"""
    D = 256
    c = _Case(cuda_device, 20_000 + K, 20_000 + K + 40, K, extra, D, mask="pre", seed=K)
    _check_ts(c, ctxs["full"], f"ncols={c.ncols} full", 1.0, tc=("tc", "presplit"))
    n1 = 2 * FLUSH * ROWS + 45                                     # one SM: 2 intervals and a partial third
    c1 = _Case(cuda_device, n1, n1 + 3 * FLUSH * ROWS, K, extra, D, mask="random", seed=K + 1)
    _check_ts(c1, ctxs["one"], f"ncols={c.ncols} one SM", -0.37, tc=("tc",))


@pytest.mark.parametrize("shape", ["reddit", "products_gf", "products_z"])
def test_production_shapes(cuda_device, ctxs, shape):
    """the Reddit-shaped hop (154 k rows, 602 features + 3 indicators + ones, D = 256: 5 chunks, 4 intervals per CTA) and
    the products-shaped heads (65 k rows, K = 104 or K = 100 with 4 indicators)"""
    n, K, extra = {"reddit": (154_007, 602, 3), "products_gf": (65_000, 104, 0), "products_z": (65_003, 100, 4)}[shape]
    D = 256
    c = _Case(cuda_device, n, n + 1000, K, extra, D, mask="pre", seed=n)
    per_half, nflush = _ts_grid(_sms(cuda_device, "full"), c.ncols, D, c.cap_n)
    if shape == "reddit":
        my = -(-(-(-n // ROWS)) // per_half)
        assert -(-my // FLUSH) >= 3, f"Reddit shape: CTA 0 walks only {my} groups"
    _check_ts(c, ctxs["full"], f"{shape} n={n} nflush={nflush}", -0.37 if shape == "reddit" else 1.0,
              tc=("tc", "presplit") if shape != "products_gf" else ("tc",))


# ---- slabs past the CTA's last interval, captured graphs ----------------------------------------------------------

def _fill_partials_nan(ctx):
    L = _L()
    p, nbytes = int(L.cdll.grapes_debug_partials(ctx)), int(L.cdll.grapes_debug_partials_bytes(ctx))
    L.grapes_fill_f32(ctx, ctypes.c_void_p(p), NAN, nbytes // 4, _st())
    torch.cuda.synchronize()


@pytest.mark.parametrize("which,n,cap_n,K", [("full", 5_017, 600_000, 104), ("full", 7_001, 400_000, 200),
                                             ("one", 3_001, 50_000, 104), ("one", 6_200, 40_000, 300)])
def test_unreached_slabs(cuda_device, ctxs, which, n, cap_n, K):
    """partial buffer filled with NaN, cap_n >> n: every CTA's nflush exceeds its intervals, and the slabs it never
    reached must be zero-filled, not read as left behind"""
    D = 256
    _fill_partials_nan(ctxs[which])
    c = _Case(cuda_device, n, cap_n, K, 2, D, mask="pre", seed=n)
    per_half, nflush = _ts_grid(_sms(cuda_device, which), c.ncols, D, cap_n)
    my = -(-(-(-n // ROWS)) // per_half)
    assert nflush > -(-my // FLUSH)
    c.check(c.run(ctxs[which], "ts", -0.37), f"{which} NaN partials n={n} cap_n={cap_n} nflush={nflush}", -0.37)
    if which == "one":                                       # k_l1_bwd_tc: 1 CTA per chunk, nflush = cap_n / 3072
        _fill_partials_nan(ctxs[which])
        c.check(c.run(ctxs[which], "tc", -0.37), f"one SM NaN partials n={n} cap_n={cap_n} [tc]", -0.37)


@pytest.mark.parametrize("kernel", ["ts", "presplit"])
def test_graph_replay_small_after_large(cuda_device, ctxs, kernel):
    """one call captured at cap_n (3 intervals per CTA of k_l1_bwd_ts, 2 of k_l1_bwd_tc), replayed with n from the device, large, small, large: each replay
    equals an eager call bit for bit and meets the float64 bound; a small n after a large one must not see the large
    replay's slabs, which stay in the same partial buffer"""
    D, K = 256, 104
    ctx = ctxs["full"]
    per_half, _ = _ts_grid(_sms(cuda_device, "full"), K + 1, D, 1 << 30)
    cap_n = 2 * FLUSH * per_half * ROWS + 7 * ROWS + 11
    c = _Case(cuda_device, cap_n, cap_n, K, 0, D, mask="pre", seed=11)
    assert _ts_grid(_sms(cuda_device, "full"), K + 1, D, cap_n)[1] == 3
    b = [_rows_for(per_half, g) for g in (96, 97, 193)]
    order = [cap_n, 33, b[2], 0, b[1], 1, cap_n, 31, b[0], cap_n + 5000, 33, b[2]]
    L = _L()
    _fill_partials_nan(ctx)
    scale = -0.37
    n_dev = torch.tensor([cap_n], dtype=torch.int32, device=cuda_device)
    grads = tuple(t.clone() for t in c.g0)
    Ya, Yb = c.presplit(ctx) if kernel == "presplit" else (c.Y, None)
    L.grapes_sampler_l1_bwd_tc(*c.args(ctx, n_dev, Ya, Yb, scale, grads))     # eager warm-up (sets the kernel attributes)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        L.grapes_sampler_l1_bwd_tc(*c.args(ctx, n_dev, Ya, Yb, scale, grads))
    for n in order:
        for dst, src in zip(grads, c.g0):
            dst.copy_(src)
        n_dev.fill_(n)
        graph.replay()
        torch.cuda.synchronize()
        eager = c.run(ctx, kernel, scale, n=n)
        assert _bits_equal(grads, eager), f"{kernel} replay n={n}: differs from an eager call"
        c.check(grads, f"{kernel} replay n={n}", scale, n=min(n, cap_n))
    del graph


# ---- rows past n -----------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("kernel", ["ts", "tc", "presplit"])
def test_rows_past_n(cuda_device, ctxs, kernel):
    """n == cap_n with cap_n % 32 != 0 (the TMA zero-fills the rest of the last group), *n_dev > cap_n (clamped to cap_n),
    and n = 0 (gradients unchanged bit for bit)"""
    D, K = 256, 131
    cap_n = 9_000 + 13
    c = _Case(cuda_device, cap_n, cap_n, K, 1, D, mask="pre", seed=5)
    c.check(c.run(ctxs["full"], kernel, 1.0), f"{kernel} n == cap_n = {cap_n}")
    c.check(c.run(ctxs["full"], kernel, 1.0, n=cap_n + 777), f"{kernel} *n_dev = cap_n + 777")
    c.check(c.run(ctxs["one"], kernel, -0.37, n=cap_n + 1), f"{kernel} one SM *n_dev = cap_n + 1", -0.37)
    for which in ("full", "one"):
        assert _bits_equal(c.run(ctxs[which], kernel, -0.37, n=0), c.g0), f"{kernel} {which}: n = 0 changed the gradients"


@pytest.mark.parametrize("mask", ["ones", "zeros"])
def test_constant_masks(cuda_device, ctxs, mask):
    """all-ones and all-zero mask words"""
    D, K = 128, 40
    c = _Case(cuda_device, 12_345, 13_000, K, 2, D, mask=mask, seed=9)
    _check_ts(c, ctxs["one"], f"mask {mask} one SM", -0.37, tc=("tc",))
    _check_ts(c, ctxs["full"], f"mask {mask}", 1.0, tc=("tc",))


# ---- accuracy where nothing cancels ----------------------------------------------------------------------------------

def test_same_sign_worst_case(cuda_device, ctxs):
    """Y >= 0, dz > 0, w2 > 0 and an all-ones mask: every product has one sign, so the truncating adds of the tensor
    core's accumulator drift one way.  k_l1_bwd_ts where every CTA runs two full 96-group intervals, and both kernels on
    one SM, where a single CTA per chunk (and half, for k_l1_bwd_ts) walks all 1563 groups: 17 intervals"""
    D, K = 256, 104
    per_half, _ = _ts_grid(_sms(cuda_device, "full"), K + 1, D, 1 << 30)
    n = 2 * FLUSH * per_half * ROWS
    c = _Case(cuda_device, n, n, K, 0, D, mask="ones", seed=21, same_sign=True)
    c1 = _Case(cuda_device, 50_000, 50_000, K, 0, D, mask="ones", seed=22, same_sign=True)
    runs = (("k_l1_bwd_ts, every CTA 2 full intervals", c, c.run(ctxs["full"], "ts")),
            ("k_l1_bwd_ts, one SM", c1, c1.run(ctxs["one"], "ts")),
            ("k_l1_bwd_tc, one SM", c1, c1.run(ctxs["one"], "tc")))
    print("\nsame-sign max |err| / mag: " + "; ".join(f"{what} {cc.worst(got):.3e}" for what, cc, got in runs))
    for what, cc, got in runs:
        cc.check(got, f"same sign: {what}")


# ---- refusals --------------------------------------------------------------------------------------------------------

def test_refusals_leave_gradients_and_context_intact(cuda_device, ctxs):
    """D = 384, ones_col < K and a partial buffer too small for nflush each return an error, write nothing, and leave
    the context usable"""
    L = _L()
    c = _Case(cuda_device, 5_000, 5_000, 104, 0, 256, mask="random", seed=4)
    n_dev = torch.tensor([c.n], dtype=torch.int32, device=cuda_device)
    for what, ctx, patch in (("D = 384", ctxs["full"], {12: 384}), ("ones_col < K", ctxs["full"], {8: c.K - 1}),
                             ("partial buffer too small", ctxs["small"], {})):
        grads = tuple(t.clone() for t in c.g0)
        a = list(c.args(ctx, n_dev, c.Y, None, 1.0, grads))
        for i, v in patch.items():
            a[i] = v
        rc = L.cdll.grapes_sampler_l1_bwd_tc(*a)
        torch.cuda.synchronize()
        assert rc != 0, f"{what}: accepted"
        assert _bits_equal(grads, c.g0), f"{what}: the gradients changed"
    small = _Case(cuda_device, 50, 64, 104, 0, 256, mask="random", seed=6)      # fits 1 MB: per_half = 2 groups
    small.check(small.run(ctxs["small"], "ts"), "small context after its refusal")
    c.check(c.run(ctxs["full"], "ts"), "full context after its refusals")
