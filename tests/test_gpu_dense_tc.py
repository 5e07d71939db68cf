"""grapes_gemm_bias_relu_tc -- H = relu(Y W^T + b) on the tcgen05 kernels, the hidden layer of the whole-graph evaluation
forward -- against float64, through the C ABI.

It is the DENSE instantiation of k_l1_fwd_ts: the sampler head's kernel with the hidden activations stored instead of
reduced against w2; it streams W through a ring of shared-memory stages (the sampler form keeps W resident when it fits:
at most 5 k-blocks of 32, K <= 160; the dense form gave wrong rows that way, which the products-shaped cases here catch).
The cases straddle the k-block counts of those forms (K <= 160, 6 to 8 k-blocks, and LONGK: more than 8 k-blocks, the
accumulator drained into an fp32 master every 8), and include a context limited to one SM, on which every CTA walks
hundreds of row tiles.  H starts as NaN: rows at or past the device count and the pitch columns [D, ldh) must keep it.  Y
carries NaN in its rows past the device count and in its pitch columns past K, which the kernel must not let into a
stored row.  The relu mask H > 0 equals, bit for bit, the maskT bits of grapes_sampler_l1_fwd_tc on the same inputs:
both instantiations compute the same pre-activation, so any difference is a bug in one epilogue."""
import ctypes

import pytest
import torch

pytestmark = pytest.mark.gpu

NAN = float("nan")
GRAPES_ERR_ARG = 1
TOL = 1e-5
D_ALL = (128, 256, 384, 512)
K_RESIDENT = (4, 15, 100, 128, 160)
K_STREAMED = (161, 192, 256)
K_LONG = (257, 288, 602, 1433)


def _L():
    from grapes_b200._lib import lib
    return lib()


def _st():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


def _r4(k):
    return (k + 3) // 4 * 4


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


def _inputs(n, cap_n, K, D, ldy, seed, dev):
    """Y [cap_n, ldy] with N(0, 1) in rows < n, columns < K and NaN everywhere else; Glorot-uniform W [D, K]; b [D]"""
    g = torch.Generator(device=dev).manual_seed(seed)
    Y = torch.full((cap_n, ldy), NAN, device=dev)
    Y[:n, :K] = torch.randn(n, K, generator=g, device=dev)
    W = (torch.rand(D, K, generator=g, device=dev) * 2 - 1) * (6.0 / (D + K)) ** 0.5
    b = torch.randn(D, generator=g, device=dev) * 0.1
    return Y, W, b


def _split(ctx, W):
    """(W_hi, W_lo, ldw) from grapes_split_tf32, ldw = round_up(K, 4)"""
    D, K = W.shape
    ldw = _r4(K)
    Wh = torch.empty((D, ldw), device=W.device)
    Wl = torch.empty((D, ldw), device=W.device)
    _L().grapes_split_tf32(ctx, _p(W), K, D, K, _p(Wh), _p(Wl), ldw, _st())
    return Wh, Wl, ldw


def _dense(ctx, Y, n_dev, cap_n, K, W, b, H, ldh):
    """grapes_gemm_bias_relu_tc into the caller's H; returns once the kernel has finished"""
    D = W.shape[0]
    Wh, Wl, ldw = _split(ctx, W)
    cnt = torch.tensor([n_dev], dtype=torch.int32, device=Y.device)
    _L().grapes_gemm_bias_relu_tc(ctx, _p(Y), Y.stride(0), _p(cnt), cap_n, K, _p(Wh), _p(Wl), ldw, D, _p(b), _p(H), ldh,
                                  _st())
    torch.cuda.synchronize()


def _mask_bits(ctx, Y, n, cap_n, K, W, b):
    """relu mask [n, D] (bool) that grapes_sampler_l1_fwd_tc (plain fp32 Y: the default k_l1_fwd_ts) emits"""
    dev = Y.device
    D = W.shape[0]
    Wh, Wl, ldw = _split(ctx, W)
    w2 = torch.randn(D, generator=torch.Generator(device=dev).manual_seed(7), device=dev)
    zpart = torch.zeros((2 * (D // 128), cap_n), device=dev)
    maskT = torch.zeros(((cap_n + 127) // 128 * 4, D), dtype=torch.int32, device=dev)
    cnt = torch.tensor([n], dtype=torch.int32, device=dev)
    _L().grapes_sampler_l1_fwd_tc(ctx, _p(Y), None, Y.stride(0), _p(cnt), cap_n, K, _p(Wh), _p(Wl), ldw, D, _p(b), _p(w2),
                                  _p(zpart), _p(maskT), _st())
    torch.cuda.synchronize()
    rows = torch.arange(n, device=dev)
    return ((maskT[rows // 32] >> (rows % 32).unsqueeze(1)) & 1).bool()


def _ref(Y, W, b, rows):
    """float64 relu(Y W^T + b) of the given rows (a slice or an index tensor), on the device"""
    K = W.shape[1]
    return torch.relu(Y[rows, :K].double() @ W.double().t() + b.double())


def _check(H, ref, rows, D, what=""):
    got = H[rows, :D]
    assert bool(torch.isfinite(got).all()), f"{what}: non-finite entries in rows < n"
    err = ((got.double() - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item()
    assert err < TOL, f"{what}: relative error {err:.3e}"


def _run_case(ctx, dev, n, cap_n, K, D, seed, ldy=None, ldh=None, n_dev=None, h_rows=None, mask=True):
    """one call at (n, cap_n, K, D) with NaN guards around everything the kernel must not write; the number of rows the
    kernel computes is min(n_dev, cap_n) (n_dev defaults to n)"""
    ldy = _r4(K) + 4 if ldy is None else ldy
    ldh = D + 4 if ldh is None else ldh
    n_dev = n if n_dev is None else n_dev
    m = min(n_dev, cap_n)
    Y, W, b = _inputs(m, cap_n, K, D, ldy, seed, dev)
    H = torch.full((h_rows or cap_n + 64, ldh), NAN, device=dev)
    _dense(ctx, Y, n_dev, cap_n, K, W, b, H, ldh)
    if m:
        _check(H, _ref(Y, W, b, slice(0, m)), slice(0, m), D, f"n={n} K={K} D={D}")
    assert bool(torch.isnan(H[m:]).all()), "a row at or past the device count was written"
    assert bool(torch.isnan(H[:, D:]).all()), "a pitch column [D, ldh) was written"
    if mask and m:
        assert torch.equal(H[:m, :D] > 0, _mask_bits(ctx, Y, m, cap_n, K, W, b)), "relu mask differs from maskT"
    return H


@pytest.mark.parametrize("D", D_ALL)
@pytest.mark.parametrize("K", K_RESIDENT + K_STREAMED + K_LONG)
def test_dense_matches_fp64(cuda_device, ctxs, K, D):
    """every form of W (resident / streamed / LONGK) at every hidden width; ldy > K with NaN pitch columns, ldh = D + 4,
    cap_n > n with NaN rows of Y behind n"""
    _run_case(ctxs["full"], cuda_device, 5000, 5200, K, D, seed=K * 7 + D)


@pytest.mark.parametrize("n", [1, 127, 128, 129, 5000, 64943])
@pytest.mark.parametrize("K,D", [(100, 256), (192, 128), (602, 512)])
def test_dense_row_counts(cuda_device, ctxs, n, K, D):
    """a partial first / last row tile, exact tile multiples and a Reddit-sized row count"""
    _run_case(ctxs["full"], cuda_device, n, n + 300, K, D, seed=n + K)


@pytest.mark.parametrize("K,D", [(100, 256), (288, 384)])
def test_dense_device_count_past_capacity(cuda_device, ctxs, K, D):
    """n_dev > cap_n: the kernel clamps to cap_n rows (the TMA map ends there) and writes no row past it"""
    _run_case(ctxs["full"], cuda_device, 3000, 3000, K, D, seed=K, n_dev=3500, h_rows=3300)


@pytest.mark.parametrize("K,D", [(100, 256), (1433, 512)])
def test_dense_zero_rows(cuda_device, ctxs, K, D):
    """n_dev = 0: every role's loop is empty; H stays NaN"""
    _run_case(ctxs["full"], cuda_device, 0, 1000, K, D, seed=3, mask=False)


@pytest.mark.parametrize("D", [128, 256, 512])
@pytest.mark.parametrize("K", [15, 100, 192, 288, 1433])
def test_dense_one_sm_persistent(cuda_device, ctxs, K, D):
    """a context limited to one SM: every CTA walks every row tile of its column half (about 390 at n = 50 000) and W
    streams through the ring whenever D > 128 (fewer SMs than column halves)"""
    _run_case(ctxs["one"], cuda_device, 50_000, 50_100, K, D, seed=K + 3 * D)


def test_dense_deterministic(cuda_device, ctxs):
    dev = cuda_device
    n, K, D = 64943, 1433, 512
    Y, W, b = _inputs(n, n, K, D, _r4(K), 11, dev)
    outs = []
    for _ in range(2):
        H = torch.full((n, D), NAN, device=dev)
        _dense(ctxs["full"], Y, n, n, K, W, b, H, D)
        outs.append(H)
    assert torch.equal(outs[0].view(torch.int32), outs[1].view(torch.int32))


def _blocks(n, step):
    for r0 in range(0, n, step):
        yield slice(r0, min(n, r0 + step))


def test_dense_products_shape(cuda_device, ctxs):
    """ogbn-products-sized hidden layer (2 449 029 rows, K = 100, D = 256), every row against float64 in row blocks"""
    dev = cuda_device
    n, K, D = 2_449_029, 100, 256
    Y, W, b = _inputs(n, n, K, D, K, 5, dev)
    H = torch.full((n + 64, D + 4), NAN, device=dev)
    _dense(ctxs["full"], Y, n, n, K, W, b, H, D + 4)
    for rows in _blocks(n, 1 << 18):
        _check(H, _ref(Y, W, b, rows), rows, D, f"rows {rows.start}..{rows.stop}")
    assert bool(torch.isnan(H[n:]).all()) and bool(torch.isnan(H[:, D:]).all())
    del Y, H
    torch.cuda.empty_cache()


def test_dense_offsets_past_2_31(cuda_device, ctxs):
    """n * ldh > 2^31 (8.5 M rows of 256: H is 8.7 GB): the element offset row * ldh of the store must not wrap.  Checked
    on 300 000 random rows and every row of the first and the last four row tiles."""
    dev = cuda_device
    n, K, D = 8_500_003, 32, 256
    assert n * D > 1 << 31
    Y, W, b = _inputs(n, n, K, D, K, 9, dev)
    H = torch.full((n + 128, D), NAN, device=dev)
    _dense(ctxs["full"], Y, n, n, K, W, b, H, D)
    g = torch.Generator(device=dev).manual_seed(1)
    rows = torch.cat([torch.arange(0, 128, device=dev), torch.randint(0, n, (300_000,), generator=g, device=dev),
                      torch.arange(n - 3 * 128 - n % 128, n, device=dev)])
    _check(H, _ref(Y, W, b, rows), rows, D, "sampled rows")
    assert bool(torch.isnan(H[n:]).all()), "a row past n was written"
    del Y, H
    torch.cuda.empty_cache()


def test_dense_refusals(cuda_device, ctxs):
    """GRAPES_ERR_ARG with the reason in grapes_last_error, and H untouched, for each layout the kernel cannot take"""
    dev = cuda_device
    L = _L()
    ctx = ctxs["full"]
    n, K, D = 300, 100, 256
    Y, W, b = _inputs(n, n, K, D, K, 2, dev)
    Wh, Wl, ldw = _split(ctx, torch.randn(640, K, device=dev))
    bb = torch.zeros(640, device=dev)
    flat = torch.full((n * (640 + 4) + 8,), NAN, device=dev)
    cnt = torch.tensor([n], dtype=torch.int32, device=dev)
    cases = {
        "D % 128 != 0": dict(D=192),
        "D > 512": dict(D=640),
        "ldh % 4 != 0": dict(ldh=D + 1),
        "H misaligned by 4 bytes": dict(off=1),
        "K > ldy": dict(K=K + 4, ldy=K),
    }
    for what, c in cases.items():
        d, k, ldh, ldy = c.get("D", D), c.get("K", K), c.get("ldh", c.get("D", D)), c.get("ldy", K)
        rc = L.cdll.grapes_gemm_bias_relu_tc(ctx, _p(Y), ldy, _p(cnt), n, k, _p(Wh), _p(Wl), ldw + 4 * (k > K), d, _p(bb),
                                             flat.data_ptr() + 4 * c.get("off", 0), ldh, _st())
        assert rc == GRAPES_ERR_ARG, f"{what}: returned {rc}"
        assert L.cdll.grapes_last_error(), what
        torch.cuda.synchronize()
        assert bool(torch.isnan(flat).all()), f"{what}: H was written"
    assert b"bad layout" in L.cdll.grapes_last_error()
