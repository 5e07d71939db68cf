"""The kernels of the classifier half of a training step and of its optimiser tail, one by one, against a float64
reference computed with torch on the CPU.

Every output buffer is pre-filled with NaN: entries a kernel must not write (rows past the device count, columns past
the width, pitch padding) are checked to still hold it, entries it documents as zeroed to be zero.  Inputs carry NaN
where the kernel must not read (rows past the device count, pitch padding).  The GEMMs run on two contexts of their
own: one with the device's SMs, which takes the 64 x 64 tiles at these shapes, and one limited to one SM, on which
the tile rule of grapes_gemm always picks the 128 x 128 tiles; both forms sum over k in the same order, so they agree
bit for bit."""
import ctypes
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F_

from dropout_utils import keep_mask

pytestmark = pytest.mark.gpu

NAN = float("nan")
GRAPES_ERR_ARG = 1
TOL = 1e-5


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _L():
    from grapes_b200._lib import lib
    return lib()


def _p(t):
    """device address of `t`; the caller keeps `t` alive until the launch is enqueued (a temporary freed earlier can
    be handed to the next allocation of the same call and overwritten before the kernel runs)"""
    return None if t is None else t.data_ptr()


def _i32(v, dev):
    return torch.tensor([v], dtype=torch.int32, device=dev)


def _rel(got, ref):
    """max |got - ref| over the scale of ref (float64)"""
    ref = ref.double()
    return ((got.double().cpu() - ref).abs().max() / ref.abs().max().clamp_min(1e-30)).item()


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
    """{"full": all SMs, "one": limited to one SM (128 x 128 GEMM tiles)}, 256 MB split-K partials each"""
    out = {"full": _new_ctx(cuda_device, 256 << 20), "one": _new_ctx(cuda_device, 256 << 20, sm_limit=1)}
    yield out
    torch.cuda.synchronize()
    for c in out.values():
        _L().cdll.grapes_ctx_destroy(c)


def _sms(dev):
    return torch.cuda.get_device_properties(dev).multi_processor_count


def _small_tiles(M_cap, N, sms):
    """the tile rule of grapes_gemm / its dropout forms: 64 x 64 tiles when the 128 x 128 grid would not cover the SMs"""
    return math.ceil(N / 128) * math.ceil(M_cap / 128) < sms


def _nan_buffer(rows, ld, dev, offset=0):
    """[rows, ld] NaN matrix; offset > 0: its base pointer sits `offset` floats past a 16-byte boundary"""
    flat = torch.full((rows * ld + offset,), NAN, dtype=torch.float32, device=dev)
    return torch.as_strided(flat, (rows, ld), (ld, 1), offset)


# ---------------------------------------------------------------------------------------------------------------------
# grapes_gemm and its dropout forms
# ---------------------------------------------------------------------------------------------------------------------
def _operand(kc, MN_dev, MN_cap, K, pad, dev, gen, offset=0):
    """(device storage with NaN past the live block, float64 live [MN_dev x K] matrix, pitch).  kc: stored [MN x K]
    K-contiguous, else [K x MN]"""
    ld = (K if kc else MN_cap) + pad
    T = _nan_buffer(MN_cap if kc else K, ld, dev, offset)
    v = torch.randn(MN_dev, K, generator=gen, dtype=torch.float64).float()
    if kc:
        T[:MN_dev, :K] = v.to(dev)
    else:
        T[:K, :MN_dev] = v.t().to(dev)
    return T, v.double(), ld


def _gemm(ctx, layout, A, lda, B, ldb, C, ldc, M_dev, M_cap, N, K, bias=None, relu=0, gate=None, ldg=0):
    _L().grapes_gemm(ctx, layout, _p(A), lda, _p(B), ldb, _p(C), ldc, _p(M_dev), M_cap, N, K, _p(bias), relu, _p(gate),
                     ldg, _stream())


GEMM_SHAPES = [(1, 1, 1, 1), (37, 30, 7, 15), (300, 257, 47, 100), (1000, 999, 256, 1433), (4100, 4097, 65, 17)]
EPILOGUES = {"plain": (False, 0, False), "bias": (True, 0, False), "bias_relu": (True, 1, False),
             "gate": (False, 0, True), "bias_relu_gate": (True, 1, True)}


@pytest.mark.parametrize("layout", [0, 1, 2, 3])
@pytest.mark.parametrize("shape", GEMM_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_gemm_matches_float64_in_both_tile_forms(cuda_device, ctxs, layout, shape):
    """C[M x N] = A B (+ bias)(relu)(gated) for every operand layout: rows < M_dev at 1e-5 of the output's scale,
    rows past M_dev and the pitch padding untouched, the 64 x 64 and 128 x 128 tile forms bit-identical."""
    dev = cuda_device
    M_cap, M, N, K = shape
    gen = torch.Generator().manual_seed(hash(shape) % 1000 + layout)
    A, a, lda = _operand(layout & 1, M, M_cap, K, 3, dev, gen)
    B, b, ldb = _operand(layout & 2, N, N, K, 5, dev, gen)
    bias64 = torch.randn(N, generator=gen, dtype=torch.float64).float().double()
    bias = bias64.float().to(dev)
    ldg = N + 2
    gate = _nan_buffer(M_cap, ldg, dev)
    g = torch.randn(M, N, generator=gen).float()
    g[g.abs() < 0.3] = 0.0                                       # exact zeros: not > 0, so gated off
    gate[:M, :N] = g.to(dev)
    M_dev = _i32(M, dev)
    prod = a @ b.t()
    assert _small_tiles(M_cap, N, _sms(dev)) and not _small_tiles(M_cap, N, 1)
    for name, (use_bias, relu, use_gate) in EPILOGUES.items():
        ref = prod + bias64 if use_bias else prod.clone()
        if relu:
            ref = ref.clamp_min(0)
        if use_gate:
            ref = torch.where(g.double() > 0, ref, torch.zeros_like(ref))
        outs = []
        for key in ("full", "one"):
            C = _nan_buffer(M_cap, N + 1, dev)
            _gemm(ctxs[key], layout, A, lda, B, ldb, C, N + 1, M_dev, M_cap, N, K, bias if use_bias else None, relu,
                  gate if use_gate else None, ldg)
            torch.cuda.synchronize()
            assert C[M:].isnan().all() and C[:, N:].isnan().all(), f"{name} {key}: wrote outside [M_dev x N]"
            assert _rel(C[:M, :N], ref) < TOL, f"{name} {key}: {_rel(C[:M, :N], ref):.2e}"
            outs.append(C[:M, :N].clone())
        assert torch.equal(outs[0], outs[1]), f"{name}: 64 x 64 and 128 x 128 tile forms differ"


@pytest.mark.parametrize("layout", [0, 1, 2, 3])
def test_gemm_unaligned_operands(cuda_device, ctxs, layout):
    """Base pointers one float past a 16-byte boundary and odd pitches: the scalar loads of load_tile / fetch_tile_s."""
    dev = cuda_device
    M_cap, M, N, K = 300, 289, 47, 37
    gen = torch.Generator().manual_seed(40 + layout)
    A, a, lda = _operand(layout & 1, M, M_cap, K, 2 if layout & 1 else 3, dev, gen, offset=1)
    B, b, ldb = _operand(layout & 2, N, N, K, 4, dev, gen, offset=1)
    assert A.data_ptr() % 16 == 4 and lda % 2 == 1 and ldb % 2 == 1
    bias64 = torch.randn(N, generator=gen).double()
    ref = (a @ b.t() + bias64).clamp_min(0)
    outs = []
    for key in ("full", "one"):
        C = _nan_buffer(M_cap, N, dev, offset=1)
        _gemm(ctxs[key], layout, A, lda, B, ldb, C, N, _i32(M, dev), M_cap, N, K, bias64.float().to(dev), 1)
        torch.cuda.synchronize()
        assert C[M:].isnan().all()
        assert _rel(C[:M], ref) < TOL, key
        outs.append(C[:M].clone())
    assert torch.equal(outs[0], outs[1])


def _drop_state(dev, seed, step):
    return torch.tensor([seed, step], dtype=torch.int64, device=dev)


@pytest.mark.parametrize("shape", [(37, 30, 7, 15), (300, 257, 47, 100), (1000, 999, 255, 63)],
                         ids=lambda s: "x".join(map(str, s)))
def test_gemm_dropout_forms(cuda_device, ctxs, shape):
    """grapes_gemm_bias_relu_dropout / grapes_gemm_gated_scaled.  Threshold 2^24 with scale 1 keeps everything: they
    equal grapes_gemm with bias + relu (layout 3) or with the gate (layout 1) bit for bit, in both tile forms.  At
    p = 0.5 the forward equals float64 relu(A W^T + b) * keep * 2 (keep = dropout_utils.keep_mask, entry row * N + col;
    N % 4 != 0 takes the unaligned keep-word path), with exact zeros where an entry was dropped."""
    dev = cuda_device
    M_cap, M, N, K = shape
    assert N % 4 != 0
    gen = torch.Generator().manual_seed(N)
    L = _L()
    A, a, lda = _operand(True, M, M_cap, K, 1, dev, gen)
    W, w, ldw = _operand(True, N, N, K, 3, dev, gen)
    Bkn, bkn, ldb = _operand(False, N, N, K, 2, dev, gen)     # [K x N] for the gated backward form
    bias64 = torch.randn(N, generator=gen).double()
    bias = bias64.float().to(dev)
    gate = _nan_buffer(M_cap, N, dev)
    g = torch.randn(M, N, generator=gen)
    g[g.abs() < 0.3] = 0.0
    gate[:M, :N] = g.to(dev)
    M_dev = _i32(M, dev)
    seed, step, tag = 12345, 7, 1
    for key in ("full", "one"):
        ctx = ctxs[key]
        # keep-all: bit-identical to the plain products
        H = _nan_buffer(M_cap, N, dev)
        Href = _nan_buffer(M_cap, N, dev)
        ds = _drop_state(dev, seed, step)
        L.grapes_gemm_bias_relu_dropout(ctx, _p(A), lda, _p(W), ldw, _p(H), N, _p(M_dev), M_cap, N, K, _p(bias), _p(ds),
                                        tag, 1 << 24, 1.0, _stream())
        _gemm(ctx, 3, A, lda, W, ldw, Href, N, M_dev, M_cap, N, K, bias, 1)
        G = _nan_buffer(M_cap, N, dev)
        Gref = _nan_buffer(M_cap, N, dev)
        L.grapes_gemm_gated_scaled(ctx, _p(A), lda, _p(Bkn), ldb, _p(G), N, _p(M_dev), M_cap, N, K, _p(gate), N, 1.0,
                                   _stream())
        _gemm(ctx, 1, A, lda, Bkn, ldb, Gref, N, M_dev, M_cap, N, K, None, 0, gate, N)
        torch.cuda.synchronize()
        assert torch.equal(H[:M], Href[:M]) and H[M:].isnan().all(), key
        assert torch.equal(G[:M], Gref[:M]) and G[M:].isnan().all(), key
        assert torch.equal(ds.cpu(), torch.tensor([seed, step])), "the GEMM forms never advance the mask counter"
        # p = 0.5
        thr = 1 << 23
        keep = torch.from_numpy(keep_mask(seed, step, tag, thr, M, N))
        assert 0.3 < keep.float().mean() < 0.7
        L.grapes_gemm_bias_relu_dropout(ctx, _p(A), lda, _p(W), ldw, _p(H), N, _p(M_dev), M_cap, N, K, _p(bias), _p(ds),
                                        tag, thr, 2.0, _stream())
        L.grapes_gemm_gated_scaled(ctx, _p(A), lda, _p(Bkn), ldb, _p(G), N, _p(M_dev), M_cap, N, K, _p(gate), N, 2.0,
                                   _stream())
        torch.cuda.synchronize()
        ref = (a @ w.t() + bias64).clamp_min(0) * keep.double() * 2
        assert _rel(H[:M], ref) < TOL, key
        assert (H[:M].cpu()[~keep] == 0).all() and H[M:].isnan().all()
        refg = torch.where(g.double() > 0, (a @ bkn.t()) * 2, torch.zeros(M, N, dtype=torch.float64))
        assert _rel(G[:M], refg) < TOL, key
        assert (G[:M].cpu()[~(g > 0)] == 0).all()


# ---------------------------------------------------------------------------------------------------------------------
# weight-gradient product and reductions
# ---------------------------------------------------------------------------------------------------------------------
def _gemm_tn_slabs(R_cap, M, N, sms):
    small = R_cap <= 16384
    t = 64 if small else 128
    slabs = max(1, (2 * sms if small else sms) // (math.ceil(N / t) * math.ceil(M / t)))
    return min(slabs, max(1, math.ceil(R_cap / 64)))


@pytest.mark.parametrize("R_cap,R", [(1000, 937), (20_000, 19_990)])
@pytest.mark.parametrize("M,N", [(1, 1), (47, 100), (100, 47), (256, 256), (1, 256)])
def test_gemm_tn_matches_float64(cuda_device, ctxs, R_cap, R, M, N):
    """out (+)= 0.5 * A[:R]^T B[:R] with NaN rows past R_dev in both operands, accumulate 0 and 1; R_cap 1000 takes
    the 64 x 64 split-K kernel, 20 000 the 128 x 128 one.  Two runs are bit-identical."""
    dev = cuda_device
    gen = torch.Generator().manual_seed(R + M + N)
    L = _L()
    A, a, lda = _operand(True, R, R_cap, M, 1, dev, gen)
    B, b, ldb = _operand(True, R, R_cap, N, 2, dev, gen)
    ref = 0.5 * (a.t() @ b)
    prior = torch.randn(M, N, generator=gen)
    R_dev = _i32(R, dev)
    for acc in (0, 1):
        runs = []
        for _ in range(2):
            out = prior.clone().to(dev) if acc else torch.full((M, N), NAN, device=dev)
            L.grapes_gemm_tn(ctxs["full"], _p(A), lda, _p(B), ldb, _p(R_dev), R_cap, M, N, 0.5, acc, _p(out),
                             _stream())
            torch.cuda.synchronize()
            runs.append(out.clone())
        want = ref + prior.double() if acc else ref
        assert _rel(runs[0], want) < TOL, f"accumulate={acc}: {_rel(runs[0], want):.2e}"
        assert torch.equal(runs[0], runs[1]), "split-K product is not deterministic"


def test_gemm_tn_refuses_a_small_partial_buffer(cuda_device):
    dev = cuda_device
    R_cap, M, N = 1000, 256, 256
    assert _gemm_tn_slabs(R_cap, M, N, _sms(dev)) * M * N * 4 > (1 << 20)
    ctx = _new_ctx(dev, 1 << 20)                                   # the smallest partial buffer a context takes
    try:
        A = torch.zeros(R_cap, M, device=dev)
        B = torch.zeros(R_cap, N, device=dev)
        out = torch.full((M, N), NAN, device=dev)
        R_dev = _i32(R_cap, dev)
        rc = _L().cdll.grapes_gemm_tn(ctx, _p(A), M, _p(B), N, _p(R_dev), R_cap, M, N, ctypes.c_float(1.0), 0,
                                      _p(out), _stream())
        torch.cuda.synchronize()
        assert rc == GRAPES_ERR_ARG and "partial buffer" in _L().last_error()
        assert out.isnan().all()
    finally:
        _L().cdll.grapes_ctx_destroy(ctx)


@pytest.mark.parametrize("C", [1, 47, 300])
@pytest.mark.parametrize("R_cap", [1, 700, 20_000])
def test_colsum_matches_float64(cuda_device, ctxs, C, R_cap):
    """out[:C] (+)= scale * sum_{r < R_dev} M[r, :C], R_dev in {0, 1, R_cap - 1}, pitch > C, NaN past R_dev and in the
    padding; out past C untouched."""
    dev = cuda_device
    gen = torch.Generator().manual_seed(C + R_cap)
    ld = C + 3
    Mx = _nan_buffer(R_cap, ld, dev)
    v = torch.randn(R_cap, C, generator=gen)
    for R in sorted({0, 1, R_cap - 1}):
        Mx[:R, :C] = v[:R].to(dev)
        R_dev = _i32(R, dev)
        ref = 0.25 * v[:R].double().sum(0)
        prior = torch.randn(C, generator=gen)
        for acc in (0, 1):
            out = torch.full((C + 4,), NAN, device=dev)
            if acc:
                out[:C] = prior.to(dev)
            _L().grapes_colsum(ctxs["full"], _p(Mx), _p(R_dev), R_cap, ld, C, 0.25, acc, _p(out), _stream())
            torch.cuda.synchronize()
            want = ref + prior.double() if acc else ref
            assert out[C:].isnan().all()
            if R == 0:
                assert torch.equal(out[:C].cpu(), want.float())
            else:
                assert _rel(out[:C], want) < TOL, f"R={R} accumulate={acc}"


@pytest.mark.parametrize("cap_n,n", [(1, 0), (1, 1), (100, 37), (3 * 4096 + 17, 3 * 4096 + 11), (5 * 4096, 5 * 4096)])
def test_vec_sum_and_fill_inv_count(cuda_device, ctxs, cap_n, n):
    """grapes_vec_sum over n spanning several 4096-element chunks, scale, divide_by_n (n = 0 gives 0), accumulate;
    grapes_fill_inv_count writes 1 / n to [0, n) and nothing past it."""
    dev = cuda_device
    L = _L()
    gen = torch.Generator().manual_seed(cap_n + n)
    v = torch.full((cap_n,), NAN, device=dev)
    x = torch.randn(n, generator=gen)
    v[:n] = x.to(dev)
    n_dev = _i32(n, dev)
    for div in (0, 1):
        for acc in (0, 1):
            out = torch.tensor([0.75 if acc else NAN], device=dev)
            L.grapes_vec_sum(ctxs["full"], _p(v), _p(n_dev), cap_n, 2.0, div, acc, _p(out), _stream())
            torch.cuda.synchronize()
            want = 2.0 * x.double().sum().item()
            if div:
                want = want / n if n > 0 else 0.0
            want += 0.75 if acc else 0.0
            got = out.item()
            scale = 2.0 * x.double().abs().sum().item() / (n if div and n else 1) + (0.75 if acc else 0.0)
            assert abs(got - want) <= TOL * scale, f"divide_by_n={div} accumulate={acc}: {got} vs {want}"
    inv = torch.full((cap_n + 3,), NAN, device=dev)
    L.grapes_fill_inv_count(ctxs["full"], _p(inv), _p(n_dev), cap_n, _stream())
    torch.cuda.synchronize()
    assert (inv[:n].cpu() == torch.tensor(1.0) / torch.tensor(float(max(n, 1)))).all()
    assert inv[n:].isnan().all()


# ---------------------------------------------------------------------------------------------------------------------
# classifier loss
# ---------------------------------------------------------------------------------------------------------------------
class _LossCase:
    """A_cap rows of logits (pitch ldl, NaN past A_dev and in the padding), B targets on a shuffled subset of the live
    rows, labels per global node (targets are node ids 3 r + 1 of a 3 B + 5 node graph)."""

    def __init__(self, dev, C, multilabel, ldl_pad, seed=0, A_cap=300, A=257, B=60):
        gen = torch.Generator().manual_seed(seed * 7919 + C * 2 + int(multilabel))
        self.C, self.A_cap, self.A, self.B, self.ldl = C, A_cap, A, B, C + ldl_pad
        l = torch.randn(A, C, generator=gen) * 3
        l[5] += 500.0
        l[6] -= 500.0
        l[7] = torch.linspace(-5e3, 5e3, C) if C > 1 else torch.tensor([5e3])       # one row with a 1e4 spread
        if multilabel:
            sat = torch.rand(A, C, generator=gen) < 0.1
            l[sat] = 100.0 * torch.sign(torch.randn(int(sat.sum()), generator=gen))   # saturated BCE logits
        self.l = l
        rest = torch.randperm(A - 8, generator=gen)[:B - 3] + 8
        ids = torch.cat([torch.tensor([5, 6, 7]), rest])            # the extreme rows are targets
        self.row_ids = ids[torch.randperm(B, generator=gen)]
        self.tgt_of_row = torch.full((A_cap,), -1, dtype=torch.int32)
        self.tgt_of_row[self.row_ids] = torch.arange(B, dtype=torch.int32)
        self.targets = torch.arange(B) * 3 + 1
        N = 3 * B + 5
        self.labels_i64 = None if multilabel else torch.randint(0, C, (N,), generator=gen)
        self.labels_f32 = (torch.rand(N, C, generator=gen) < 0.3).float() if multilabel else None
        self.dev = dev

    def device_args(self):
        d = self.dev
        logits = _nan_buffer(self.A_cap, self.ldl, d)
        logits[:self.A, :self.C] = self.l.to(d)
        return dict(logits=logits, A_dev=_i32(self.A, d), row_ids=self.row_ids.to(torch.int32).to(d),
                    tgt_of_row=self.tgt_of_row.to(d), targets=self.targets.to(torch.int32).to(d),
                    labels_i64=None if self.labels_i64 is None else self.labels_i64.to(d),
                    labels_f32=None if self.labels_f32 is None else self.labels_f32.to(d))

    def reference(self, reg, keep=None, scale=1.0):
        """float64 autograd of the reference's loss (main.py:260-261) + reg * var(l[:A], dim=1).sum(), on the dropped
        logits when `keep` is given; the gradient is w.r.t. the logits before dropout"""
        l = self.l.double().requires_grad_(True)
        ld = l * keep.double() * scale if keep is not None else l
        lt = ld[self.row_ids]
        if self.labels_i64 is not None:
            loss = F_.cross_entropy(lt, self.labels_i64[self.targets])
        else:
            loss = F_.binary_cross_entropy_with_logits(lt, self.labels_f32[self.targets].double())
        if reg:
            loss = loss + reg * torch.var(ld, dim=1).sum()
        loss.backward()
        return loss.item(), l.grad, ld.detach()


def _run_loss(ctx, case, args, form, reg, drop=None):
    """form "rows": the row-parallel form (tgt_of_row given, C <= 1024); "targets": the target-row form"""
    d = case.dev
    dl = _nan_buffer(case.A_cap, case.ldl, d)
    loss = torch.full((1,), NAN, device=d)
    colsum = torch.full((case.C + 2,), NAN, device=d)
    common = (ctx, _p(args["logits"]), case.ldl, case.C, _p(args["A_dev"]), case.A_cap, _p(args["row_ids"]),
              _p(args["tgt_of_row"]) if form == "rows" else None, _p(args["targets"]), case.B, _p(args["labels_i64"]),
              _p(args["labels_f32"]), reg, _p(dl), _p(loss), _p(colsum))
    if drop is None:
        _L().grapes_classifier_loss(*common, _stream())
    else:
        state, thr, scale = drop
        _L().grapes_classifier_loss_dropout(*common, _p(state), 2, thr, scale, _stream())
    torch.cuda.synchronize()
    return dl, loss.item(), colsum


def _check_loss(case, form, dl, loss, colsum, ref_loss, ref_grad):
    A, C = case.A, case.C
    assert abs(loss - ref_loss) <= TOL * abs(ref_loss) + 1e-12, f"{form}: loss {loss} vs {ref_loss}"
    assert _rel(dl[:A, :C], ref_grad) < TOL, f"{form}: dlogits {_rel(dl[:A, :C], ref_grad):.2e}"
    ref_cs = ref_grad.sum(0)
    assert (colsum[:C].double().cpu() - ref_cs).abs().max() <= TOL * max(ref_cs.abs().max().item(),
                                                                         ref_grad.abs().max().item()), f"{form}: colsum"
    assert colsum[C:].isnan().all()
    if form == "rows":          # the row-parallel form writes rows < A_dev, columns < C only
        assert dl[A:].isnan().all() and dl[:A, C:].isnan().all()
    else:                       # the target-row form zeroes A_cap rows of pitch ldl first
        assert (dl[A:] == 0).all() and (dl[:A, C:] == 0).all()


LOSS_C = [1, 2, 47, 172, 1024, 1025, 1500]


@pytest.mark.parametrize("C", LOSS_C)
@pytest.mark.parametrize("multilabel", [False, True], ids=["ce", "bce"])
@pytest.mark.parametrize("reg", [0.0, 0.1])
@pytest.mark.parametrize("ldl_pad", [0, 3])
def test_classifier_loss_both_forms(cuda_device, ctxs, C, multilabel, reg, ldl_pad):
    """grapes_classifier_loss: loss at 1e-5 relative, dlogits[:A] and the column sums at 1e-5 of their scale, rows past
    A_dev as each form documents, the two forms' dlogits bit-identical where both apply (C <= 1024).  Above C = 1024
    the call takes the target-row form even with tgt_of_row given."""
    if C == 1 and reg:
        pytest.skip("the unbiased variance of one element is NaN in the reference; the kernel drops the term at C = 1")
    case = _LossCase(cuda_device, C, multilabel, ldl_pad)
    ref_loss, ref_grad, _ = case.reference(reg)
    args = case.device_args()
    forms = ("rows", "targets") if C <= 1024 else ("targets",)
    got = {}
    for form in forms:
        dl, loss, colsum = _run_loss(ctxs["full"], case, args, form, reg)
        _check_loss(case, form, dl, loss, colsum, ref_loss, ref_grad)
        got[form] = dl[:case.A, :C].clone()
    if C > 1024:            # tgt_of_row given but ignored: same result as the target-row call, zeroed padding included
        dl, loss, colsum = _run_loss(ctxs["full"], case, args, "rows", reg)
        _check_loss(case, "targets", dl, loss, colsum, ref_loss, ref_grad)
    else:
        assert torch.equal(got["rows"], got["targets"]), "the two loss forms' dlogits differ"
    assert torch.equal(args["logits"][:case.A, :C].cpu(), case.l), "the plain loss must not write the logits"


@pytest.mark.parametrize("C", [2, 47, 1024, 1025])
@pytest.mark.parametrize("multilabel", [False, True], ids=["ce", "bce"])
@pytest.mark.parametrize("reg", [0.0, 0.1])
def test_classifier_loss_dropout(cuda_device, ctxs, C, multilabel, reg):
    """grapes_classifier_loss_dropout.  p = 0 (threshold 2^24, scale 1): loss, dlogits and column sums equal
    grapes_classifier_loss bit for bit and the logits stay as they were.  p = 0.5: float64 on the dropped logits, the
    logits written back dropped, dlogits = d loss / d (pre-dropout logits).  Every call advances drop_state[1] by one."""
    dev = cuda_device
    case = _LossCase(dev, C, multilabel, 3, seed=1)
    seed, step = 99, 3
    forms = ("rows", "targets") if C <= 1024 else ("targets",)
    for form in forms:
        # p = 0
        args = case.device_args()
        plain = _run_loss(ctxs["full"], case, args, form, reg)
        state = _drop_state(dev, seed, step)
        dl, loss, colsum = _run_loss(ctxs["full"], case, args, form, reg, drop=(state, 1 << 24, 1.0))
        assert int(state[1]) == step + 1 and int(state[0]) == seed, form
        assert torch.equal(dl[:case.A, :C], plain[0][:case.A, :C]) and loss == plain[1], form
        assert torch.equal(colsum[:C], plain[2][:C]), form
        assert torch.equal(args["logits"][:case.A, :C].cpu(), case.l), form
        # p = 0.5
        thr = 1 << 23
        keep = torch.from_numpy(keep_mask(seed, step + 1, 2, thr, case.A, C))
        ref_loss, ref_grad, ref_dropped = case.reference(reg, keep, 2.0)
        dl, loss, colsum = _run_loss(ctxs["full"], case, args, form, reg, drop=(state, thr, 2.0))
        assert int(state[1]) == step + 2, form
        _check_loss(case, form, dl, loss, colsum, ref_loss, ref_grad)
        assert torch.equal(args["logits"][:case.A, :C].cpu().double(), ref_dropped), f"{form}: logits not written dropped"
        assert args["logits"][case.A:].isnan().all()
        assert (dl[:case.A, :C].cpu()[~keep] == 0).all()


# ---------------------------------------------------------------------------------------------------------------------
# argmax, Adam, GFlowNet loss
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C", [1, 31, 32, 33, 172, 1025])
def test_argmax_rows(cuda_device, ctxs, C):
    """grapes_argmax_rows against torch.argmax: exact ties go to the lowest column (columns 3 and 35 share a lane, 3 and
    36 do not), a row of -inf gives 0, repeated row ids, outputs past B_dev untouched.  NaN never wins -- the kernel's
    documented rule, which is NOT torch's (torch.argmax returns the NaN's column): a NaN entry is skipped, and a row
    of NaN only gives 0."""
    dev = cuda_device
    gen = torch.Generator().manual_seed(C)
    R, ldl = 40, C + 1
    l = torch.randn(R, C, generator=gen)
    l[0] = -math.inf
    if C > 36:
        l[1, 3] = l[1, 35] = l[1].max() + 1.0
        l[2, 3] = l[2, 36] = l[2].max() + 1.0
        l[3, 36] = l[3, 35] = l[3].max() + 1.0                  # tie across lanes, the higher lane first in memory order
    if C > 1:
        l[4, C - 1] = NAN
        l[4, C // 2] = 1e30                                      # NaN in the row: the finite maximum wins
        l[5, 0] = NAN
    l[6] = NAN
    l[7] = 2.0                                                   # the whole row tied
    logits = _nan_buffer(R, ldl, dev)
    logits[:, :C] = l.to(dev)
    row_ids = torch.tensor([0, 1, 2, 3, 4, 5, 6, 7, 1, 1, 8, 39, 7, 20, 0], dtype=torch.int32)
    B, cap_B = int(row_ids.numel()), int(row_ids.numel()) + 5
    out = torch.full((cap_B,), -7, dtype=torch.int32, device=dev)
    rows_dev, B_dev = row_ids.to(dev), _i32(B, dev)
    _L().grapes_argmax_rows(ctxs["full"], _p(logits), ldl, C, _p(rows_dev), _p(B_dev), cap_B, _p(out),
                            _stream())
    torch.cuda.synchronize()
    rows = l[row_ids.long()]
    ref = torch.argmax(torch.nan_to_num(rows, nan=-math.inf), dim=1)
    assert torch.equal(out[:B].cpu().long(), ref)
    assert (out[B:] == -7).all()
    if C > 36:
        assert out[1].item() == 3 and out[2].item() == 3 and out[3].item() == 35
    assert out[0].item() == 0 and out[6].item() == 0 and out[7].item() == 0


def _adam_case(dev, n0, n1, gap=1000, head=17, tail=23):
    off0 = head
    off1 = off0 + n0 + gap
    n = off1 + n1 + tail
    return off0, off1, n


@pytest.mark.parametrize("n0,n1", [((1 << 20) + 3, (1 << 20) + 7), (0, 5000), (4099, 0)])
def test_adam_step2_matches_torch_adam(cuda_device, ctxs, n0, n1):
    """grapes_adam_step2 against torch.optim.Adam(foreach=False) with two groups (lr 1e-3 and 1e-4), 20 steps, gradients
    from 1e-12 to 1e3 with exact zeros: weights at rtol 1e-6 / atol 1e-7 of float32 torch, entries outside the groups
    untouched, and each group's step count advanced exactly once per call (the last-block ticket resets), only for a
    group that has entries."""
    dev = cuda_device
    L = _L()
    gen = torch.Generator().manual_seed(n0 + 3 * n1)
    off0, off1, n = _adam_case(dev, n0, n1)
    p0 = torch.randn(n, generator=gen)
    groups = [(off0, n0, 1e-3), (off1, n1, 1e-4)]
    ref = [torch.nn.Parameter(p0[o:o + k].clone()) for o, k, _ in groups]
    opt = torch.optim.Adam([{"params": [ref[0]], "lr": 1e-3}, {"params": [ref[1]], "lr": 1e-4}], foreach=False)
    p = p0.clone().to(dev)
    m = torch.full((n,), 0.0, device=dev)
    v = torch.full((n,), 0.0, device=dev)
    live = torch.zeros(n, dtype=torch.bool)
    for o, k, _ in groups:
        live[o:o + k] = True
    canary_p = p0[~live].clone()
    m[~live.to(dev)] = 3.0
    v[~live.to(dev)] = 5.0
    steps = torch.zeros(2, device=dev)
    g = torch.zeros(n)
    for i in range(20):
        g = torch.randn(n, generator=gen) * torch.pow(10.0, torch.rand(n, generator=gen) * 15 - 12)
        g[torch.rand(n, generator=gen) < 0.05] = 0.0
        g[~live] = NAN                                           # never read
        for r, (o, k, _) in zip(ref, groups):
            r.grad = g[o:o + k].clone()
        opt.step()
        g_dev = g.to(dev)
        L.grapes_adam_step2(ctxs["full"], _p(p), _p(g_dev), _p(m), _p(v), off0, n0, 1e-3, off1, n1, 1e-4, 0.9, 0.999,
                            1e-8, _p(steps), _stream())
        torch.cuda.synchronize()
        assert steps.tolist() == [float(i + 1) if n0 else 0.0, float(i + 1) if n1 else 0.0], f"call {i}: {steps.tolist()}"
    pc = p.cpu()
    for r, (o, k, _) in zip(ref, groups):
        torch.testing.assert_close(pc[o:o + k], r.detach(), rtol=1e-6, atol=1e-7)
    assert torch.equal(pc[~live], canary_p)
    assert (m.cpu()[~live] == 3.0).all() and (v.cpu()[~live] == 5.0).all()


@pytest.mark.parametrize("reinforce", [0, 1])
@pytest.mark.parametrize("have_log_z", [0, 1])
def test_gfn_finalize_closed_forms(cuda_device, ctxs, reinforce, have_log_z):
    """grapes_gfn_finalize / grapes_gfn_finalize_scale against main.py:271-282 in float64: log_z = mean(gcn_z logits)
    - log_z_init (0 without the gcn_z net); REINFORCE: loss_gfn = -tot * loss_c, gradient scales (-loss_c, 0); trajectory
    balance: r = log_z + tot + coef * loss_c, loss_gfn = r^2, gradient scales (2 r, 2 r); grad = scale * direction."""
    dev = cuda_device
    L = _L()
    loss_c, tot, log_z_mean, coef, log_z_init = 1.7320508, -35.25, 0.3125, 1e4, -0.5
    log_z = (log_z_mean - log_z_init) if have_log_z else 0.0
    if reinforce:
        want = dict(loss_gfn=-tot * loss_c, g_gf=-loss_c, g_z=0.0)
    else:
        r = log_z + tot + coef * loss_c
        want = dict(loss_gfn=r * r, g_gf=2 * r, g_z=2 * r)
    idx = dict(log_z=3, loss_gfn=4, g_gf=5, g_z=6)
    gen = torch.Generator().manual_seed(5)
    dir_gf, dir_z = torch.randn(1000, generator=gen), torch.randn(300, generator=gen)
    dgf, dz = dir_gf.to(dev), dir_z.to(dev)
    for fused in (False, True):
        scal = torch.full((16,), NAN, device=dev)
        scal[0], scal[1], scal[2] = loss_c, tot, log_z_mean
        inputs = scal[:3].double().cpu()
        grad_gf = torch.full((1001,), NAN, device=dev)
        grad_z = torch.full((301,), NAN, device=dev)
        if fused:
            L.grapes_gfn_finalize_scale(ctxs["full"], _p(scal), coef, log_z_init, reinforce, have_log_z,
                                        _p(dgf), 1000, _p(grad_gf), _p(dz), 300, _p(grad_z),
                                        _stream())
        else:
            L.grapes_gfn_finalize(ctxs["full"], _p(scal), coef, log_z_init, reinforce, have_log_z, _stream())
        torch.cuda.synchronize()
        s = scal.double().cpu()
        assert torch.equal(s[:3], inputs)
        lz = (inputs[2].item() - np.float32(log_z_init)) if have_log_z else 0.0
        assert abs(s[idx["log_z"]].item() - lz) <= 1e-6 * max(1.0, abs(lz))
        for k in ("loss_gfn", "g_gf", "g_z"):
            assert abs(s[idx[k]].item() - want[k]) <= 1e-6 * max(1.0, abs(want[k])), f"{k}: {s[idx[k]].item()} vs {want[k]}"
        assert s[7:].isnan().all()
        if fused:
            assert _rel(grad_gf[:1000], want["g_gf"] * dir_gf.double()) < TOL and grad_gf[1000:].isnan().all()
            if want["g_z"] == 0.0:
                assert (grad_z[:300] == 0).all()
            else:
                assert _rel(grad_z[:300], want["g_z"] * dir_z.double()) < TOL
            assert grad_z[300:].isnan().all()
