"""The kernels of one sampler hop (main.py:180-213 and the backward of its width-1 aggregation), one by one through the
C ABI, against exact integer references and float64, on a DIRECTED graph (directed_utils.directed_synth).

Integer outputs match exactly; float outputs hold 1e-5 relative to the largest magnitude of the float64 reference.
Outputs are pre-filled with -1 / NaN so that an unwritten entry fails; device counts sit below the capacities, with
finite junk in the input rows past them.  Every documented precondition is kept: cnt_scratch is all zero on entry, and
the graph's context is created with max_frontier above every capacity passed."""
import numpy as np
import pytest
import torch

from directed_utils import directed_synth
from oracle import reference_port as rp
from parity_utils import TOL, _rel

pytestmark = pytest.mark.gpu

NAN = float("nan")


def _L():
    from grapes_b200._lib import lib
    return lib()


def _st():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return None if t is None else t.data_ptr()


def _i32(v, dev):
    return torch.tensor([v], dtype=torch.int32, device=dev)


def _pack(mask: torch.Tensor, W: int) -> torch.Tensor:
    """bool [N] -> int32 bitmap words [W] (bit v & 31 of word v >> 5)"""
    b = np.zeros(W * 32, dtype=bool)
    b[:mask.numel()] = mask.cpu().numpy()
    return torch.from_numpy(np.packbits(b, bitorder="little").view(np.int32).copy())


def _unpack(words: torch.Tensor, N: int) -> torch.Tensor:
    return torch.from_numpy(np.unpackbits(words.cpu().numpy().view(np.uint8), bitorder="little")[:N].astype(bool))


@pytest.fixture(scope="module")
def graph(cuda_device):
    """Directed power-law graph: hub rows with hundreds of out-edges, a fifth of the nodes without any, destinations
    of more than 32 in-edges inside one hop."""
    from grapes_b200.graph import DeviceGraph
    d = directed_synth("small", 6, power_law=1.5)
    adj = rp.build_adjacency(d.edge_index, d.num_nodes)
    g = DeviceGraph.from_edge_index(d.edge_index, d.num_nodes, device=cuda_device, max_frontier=1 << 20)
    assert np.array_equal(g.indptr.cpu().numpy(), adj.indptr) and np.array_equal(g.indices.cpu().numpy(), adj.indices)
    return d, adj, g


def _rows(d, adj):
    """a row list with rows without out-edges first, consecutive and last, and the hub row"""
    deg = torch.from_numpy(adj.indptr[1:] - adj.indptr[:-1])
    empty = (deg == 0).nonzero().squeeze(1)
    hub = int(deg.argmax())
    tr = d.train_mask.nonzero().squeeze(1)
    tr = tr[~torch.isin(tr, torch.cat([empty[:4], torch.tensor([hub])]))][:128]
    rows = torch.cat([empty[:3], torch.tensor([hub]), tr, empty[3:4]])
    assert int(deg[hub]) > 500
    return rows


def _expand(g, rows, cap_P, cap_m, dev):
    L = _L()
    P = rows.numel()
    r = torch.full((cap_P,), 7, dtype=torch.int32, device=dev)          # finite junk past P
    r[:P] = rows.to(dev, torch.int32)
    out = dict(rows=r, P=_i32(P, dev), row_off=torch.full((cap_P + 1,), -1, dtype=torch.int32, device=dev),
               m=_i32(-1, dev), e_row=torch.full((cap_m,), -1, dtype=torch.int32, device=dev),
               e_col=torch.full((cap_m,), -1, dtype=torch.int32, device=dev),
               bm_rows=torch.zeros(g.num_words, dtype=torch.int32, device=dev),
               bm_batch=torch.zeros(g.num_words, dtype=torch.int32, device=dev),
               ovf=torch.zeros(1, dtype=torch.int32, device=dev))
    L.grapes_expand_frontier(g.ctx, _p(g.indptr), _p(g.indices), _p(r), _p(out["P"]), cap_P, _p(out["row_off"]),
                             _p(out["m"]), cap_m, _p(out["e_row"]), _p(out["e_col"]), _p(out["bm_rows"]),
                             _p(out["bm_batch"]), _p(out["ovf"]), _st())
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("cap_P", [200, 9000])          # k_expand_fused (cap_P <= 8192) and the two-kernel form
def test_expand_frontier(cuda_device, graph, cap_P):
    d, adj, g = graph
    N = d.num_nodes
    for rows in (_rows(d, adj), torch.zeros(0, dtype=torch.int64)):
        P = rows.numel()
        ex = _expand(g, rows, cap_P, 1 << 16, cuda_device)
        assert int(ex["ovf"].item()) == 0
        deg = torch.from_numpy(adj.indptr[1:] - adj.indptr[:-1])
        ref_off = torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(deg[rows], 0)])
        assert torch.equal(ex["row_off"][:P + 1].cpu().long(), ref_off), "row_off"
        m = int(ex["m"].item())
        assert m == int(ref_off[-1]), "*m"
        nh = rp.get_neighborhoods(rows, adj)
        pos = torch.repeat_interleave(torch.arange(P), deg[rows])
        assert torch.equal(ex["e_row"][:m].cpu().long(), pos), "e_row"
        assert torch.equal(ex["e_col"][:m].cpu().long(), nh[1]), "e_col"
        want_rows = torch.zeros(N, dtype=torch.bool)
        want_rows[rows] = True
        want_batch = torch.zeros(N, dtype=torch.bool)
        want_batch[rows[deg[rows] > 0]] = True
        want_batch[nh[1]] = True
        assert torch.equal(_unpack(ex["bm_rows"], N), want_rows), "bm_rows"
        assert torch.equal(_unpack(ex["bm_batch"], N), want_batch), "bm_batch"


def _rank_ref(bb, bp, W):
    batch = bb.nonzero().squeeze(1)
    nbm = bb & ~bp
    nb = nbm.nonzero().squeeze(1)
    words_b = _pack(bb, W).numpy().view(np.uint32)
    words_n = _pack(nbm, W).numpy().view(np.uint32)
    pop = lambda w: torch.from_numpy(np.unpackbits(w.view(np.uint8)).reshape(-1, 32).sum(1).astype(np.int64))
    pb, pn = pop(words_b), pop(words_n)
    pref_b = torch.cumsum(pb, 0) - pb
    pref_n = torch.cumsum(pn, 0) - pn
    nb_local = torch.searchsorted(batch, nb)
    nb_index = torch.full((batch.numel(),), -1, dtype=torch.int64)
    nb_index[nb_local] = torch.arange(nb.numel())
    return batch, nb, nb_local, nb_index, pref_b, pref_n, nbm


@pytest.mark.parametrize("N,hop", [(300_007, 0), (300_007, 3), (300_007, 6), (1_000_003, 6), (1_000, 3)])
def test_rank_nodes(cuda_device, N, hop):
    """Decoupled look-back over many 1024-word tiles; indicator columns of 8 rows: columns h < hop come from bm_ind,
    column hop is the candidate mask (also written to bm_ind row hop), the last column is bm_ind's last row."""
    from grapes_b200.graph import DeviceGraph
    dev = cuda_device
    L = _L()
    g = DeviceGraph(torch.zeros(N + 1, dtype=torch.int64, device=dev), torch.zeros(0, dtype=torch.int32, device=dev), N)
    W, R = g.num_words, 8
    gen = torch.Generator().manual_seed(N + hop)
    cases = [(torch.rand(N, generator=gen) < 0.3, torch.rand(N, generator=gen) < 0.1),
             (torch.zeros(N, dtype=torch.bool), torch.zeros(N, dtype=torch.bool))]           # empty bitmap
    bb = torch.rand(N, generator=gen) < 0.05
    cases.append((bb, bb | (torch.rand(N, generator=gen) < 0.05)))                          # prev covers batch: c = 0
    for bb, bp in cases:
        batch, nb, nb_local, nb_index, pref_b, pref_n, nbm = _rank_ref(bb, bp, W)
        n, c = batch.numel(), nb.numel()
        cap_n = n + 33
        ind_in = torch.rand(R, N, generator=gen) < 0.5
        bm_ind = torch.stack([_pack(ind_in[h], W) for h in range(R)]).to(dev)
        o = {k: torch.full((cap_n,), -1, dtype=torch.int32, device=dev)
             for k in ("batch_nodes", "nb_nodes", "nb_local", "nb_index", "ind_bits")}
        pref_batch = torch.full((W + 1,), -1, dtype=torch.int32, device=dev)
        pref_nb = torch.full((W + 1,), -1, dtype=torch.int32, device=dev)
        n_dev, c_dev, ovf = _i32(-1, dev), _i32(-1, dev), torch.zeros(1, dtype=torch.int32, device=dev)
        bm_batch, bm_prev = _pack(bb, W).to(dev), _pack(bp, W).to(dev)
        L.grapes_rank_nodes(g.ctx, _p(bm_batch), _p(bm_prev), _p(pref_batch), _p(pref_nb),
                            _p(o["batch_nodes"]), _p(o["nb_nodes"]), _p(o["nb_local"]), _p(o["nb_index"]),
                            _p(o["ind_bits"]), _p(bm_ind), R, hop, cap_n, _p(n_dev), _p(c_dev), _p(ovf), _st())
        torch.cuda.synchronize()
        assert int(ovf.item()) == 0 and int(n_dev.item()) == n and int(c_dev.item()) == c, "n / c"
        assert torch.equal(pref_batch[:W].cpu().long(), pref_b), "pref_batch"
        assert torch.equal(pref_nb[:W].cpu().long(), pref_n), "pref_nb"
        assert torch.equal(o["batch_nodes"][:n].cpu().long(), batch), "batch_nodes"
        assert torch.equal(o["nb_nodes"][:c].cpu().long(), nb), "nb_nodes"
        assert torch.equal(o["nb_local"][:c].cpu().long(), nb_local), "nb_local"
        assert torch.equal(o["nb_index"][:n].cpu().long(), nb_index), "nb_index"
        assert bool((o["batch_nodes"][n:] == -1).all() and (o["nb_nodes"][c:] == -1).all()), "written past the count"
        want = torch.zeros(n, dtype=torch.int64)
        for h in range(R):
            if h < R - 1 and h < hop:
                col = ind_in[h][batch]
            elif h == hop:
                col = nbm[batch]
            elif h == R - 1:
                col = ind_in[R - 1][batch]
            else:
                continue
            want |= col.long() << h
        assert torch.equal(o["ind_bits"][:n].cpu().long() & 0xff, want), "ind_bits"
        got_ind = bm_ind.cpu()
        for h in range(R):
            want_row = _pack(nbm, W) if h == hop else _pack(ind_in[h], W)
            assert torch.equal(got_ind[h], want_row), f"bm_ind row {h}"


def _hop_structure(g, adj, rows, dev, cap_n=None):
    """expansion + rank + local edges of one hop (the engine's order), with the float64-independent references"""
    L = _L()
    N = adj.shape[0]
    ex = _expand(g, rows, 256, 1 << 16, dev)
    W = g.num_words
    nh = rp.get_neighborhoods(rows, adj)
    bb = torch.zeros(N, dtype=torch.bool)
    bb[nh.view(-1)] = True
    bp = torch.zeros(N, dtype=torch.bool)
    bp[rows] = True
    batch, nb, nb_local, nb_index, pref_b, pref_n, nbm = _rank_ref(bb, bp, W)
    n = batch.numel()
    cap_n = n + 37 if cap_n is None else cap_n
    assert cap_n > n
    h = dict(ex=ex, n=n, cap_n=cap_n, batch=batch, m=nh.shape[1], cap_m=1 << 16, nh=nh, nb=nb, nb_local=nb_local,
             nb_index=nb_index,
             pref_batch=torch.zeros(W + 1, dtype=torch.int32, device=dev),
             batch_nodes=torch.full((cap_n,), 5, dtype=torch.int32, device=dev),
             n_dev=_i32(-1, dev), ovf=torch.zeros(1, dtype=torch.int32, device=dev))
    L.grapes_rank_nodes(g.ctx, _p(ex["bm_batch"]), _p(ex["bm_rows"]), _p(h["pref_batch"]), None,
                        _p(h["batch_nodes"]), None, None, None, None, None, 0, 0, cap_n, _p(h["n_dev"]), None,
                        _p(h["ovf"]), _st())
    torch.cuda.synchronize()
    assert int(h["n_dev"].item()) == n
    h["src_ref"] = torch.searchsorted(batch, nh[0])
    h["dst_ref"] = torch.searchsorted(batch, nh[1])
    return h


def _csr_ref(key, val, n):
    keep = key != val
    key, val = key[keep], val[keep]
    order = torch.argsort(key * n + val, stable=True)
    cnt = torch.bincount(key, minlength=n)
    off = torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(cnt, 0)])
    dinv = 1.0 / torch.sqrt(cnt.float() + 1.0)
    return off, val[order], dinv, int(keep.sum())


@pytest.mark.parametrize("form", ["hist_done", "single_cta", "multi_launch"])
def test_edges_to_local_and_build_csr(cuda_device, graph, form):
    d, adj, g = graph
    dev = cuda_device
    L = _L()
    rows = _rows(d, adj)
    h = _hop_structure(g, adj, rows, dev, cap_n={"hist_done": None, "single_cta": 4096, "multi_launch": 8000}[form])
    n, cap_n, cap_m, ex = h["n"], h["cap_n"], h["cap_m"], h["ex"]
    e_src = torch.full((cap_m,), -1, dtype=torch.int32, device=dev)
    e_dst = torch.full((cap_m,), -1, dtype=torch.int32, device=dev)
    cnt = torch.zeros(cap_n, dtype=torch.int32, device=dev)
    L.grapes_edges_to_local(g.ctx, _p(ex["rows"]), _p(ex["e_row"]), _p(ex["e_col"]), _p(ex["m"]), cap_m,
                            _p(ex["bm_batch"]), _p(h["pref_batch"]), cap_n, _p(e_src), _p(e_dst),
                            _p(cnt) if form == "hist_done" else None, _st())
    torch.cuda.synchronize()
    m = h["m"]
    assert torch.equal(e_src[:m].cpu().long(), h["src_ref"]) and torch.equal(e_dst[:m].cpu().long(), h["dst_ref"])
    off_ref, val_ref, dinv_ref, nnz_ref = _csr_ref(h["dst_ref"], h["src_ref"], n)
    assert int(off_ref[1:].sub(off_ref[:-1]).max()) > 32, "no row takes the rank-sort path"
    off = torch.full((cap_n + 1,), -1, dtype=torch.int32, device=dev)
    sval = torch.full((cap_m,), -1, dtype=torch.int32, device=dev)
    tmp = torch.empty(cap_m, dtype=torch.int32, device=dev)
    dinv = torch.full((cap_n,), NAN, device=dev)
    nnz = _i32(-1, dev)
    L.grapes_build_csr(g.ctx, _p(e_dst), _p(e_src), _p(ex["m"]), cap_m, _p(h["n_dev"]), cap_n, _p(cnt),
                       int(form == "hist_done"), _p(off), _p(sval), _p(tmp), _p(dinv), _p(nnz), _p(h["ovf"]), _st())
    torch.cuda.synchronize()
    assert int(h["ovf"].item()) == 0
    assert int(nnz.item()) == nnz_ref, "nnz"
    assert torch.equal(off[:n + 1].cpu().long(), off_ref), "off"
    assert torch.equal(sval[:nnz_ref].cpu().long(), val_ref), "sorted_val"
    assert torch.equal(dinv[:n].cpu(), dinv_ref), "dinv"
    assert int(cnt.abs().sum()) == 0, "cnt_scratch not all zero again"


def _hop_csr(g, adj, rows, dev):
    h = _hop_structure(g, adj, rows, dev)
    off, val, dinv, nnz = _csr_ref(h["dst_ref"], h["src_ref"], h["n"])
    cap_n = h["cap_n"]
    pad = lambda t, fill, dt: torch.cat([t.to(dt), torch.full((cap_n + 1 - t.numel(),), fill, dtype=dt)]).to(dev)
    h.update(in_off=pad(off, off[-1].item(), torch.int32), in_src=val.to(dev, torch.int32),
             dinv=torch.cat([dinv, torch.full((cap_n - h["n"],), 0.75)]).to(dev), dinv_ref=dinv.double(),
             off_ref=off, val_ref=val)
    return h


def _agg_ref(z, off, val, dinv, bias):
    n = dinv.numel()
    dst = torch.repeat_interleave(torch.arange(n), off[1:] - off[:-1])
    return (dinv * dinv * z[:n]).index_add(0, dst, dinv[val] * dinv[dst] * z[val]) + bias


@pytest.mark.parametrize("nparts", [1, 2, 4])
@pytest.mark.parametrize("with_bias", [False, True])
def test_aggregate_scalar(cuda_device, graph, nparts, with_bias):
    d, adj, g = graph
    dev = cuda_device
    h = _hop_csr(g, adj, _rows(d, adj), dev)
    n, cap_n = h["n"], h["cap_n"]
    gen = torch.Generator().manual_seed(nparts)
    z = torch.randn(nparts, cap_n, generator=gen)
    zd = z.to(dev)
    bias = torch.tensor([0.625], device=dev) if with_bias else None
    out = torch.full((cap_n,), NAN, device=dev)
    zero = torch.full((cap_n,), NAN, device=dev)
    _L().grapes_aggregate_scalar(g.ctx, _p(zd), nparts, cap_n, _p(h["n_dev"]), cap_n, _p(h["in_off"]), _p(h["in_src"]),
                                 _p(h["dinv"]), _p(bias), _p(out), _p(zero), _st())
    torch.cuda.synchronize()
    ref = _agg_ref(z.double().sum(0), h["off_ref"], h["val_ref"], h["dinv_ref"], 0.625 if with_bias else 0.0)
    assert _rel(out[:n], ref) < TOL
    assert bool(torch.isnan(out[n:]).all()), "written past n"
    assert bool((zero[:n] == 0).all()) and bool(torch.isnan(zero[n:]).all()), "zero_out"


@pytest.mark.parametrize("fused", [True, False])
def test_aggregate_scalar_T(cuda_device, graph, fused):
    """dz = A_hat^T dl on a hop graph whose expanded rows include rows without out-edges that are frontier nodes
    (another row points to them): every dz[j], j < n, must be written -- those rows with dinv[j]^2 dl[j]."""
    d, adj, g = graph
    dev = cuda_device
    rows = _rows(d, adj)
    h = _hop_csr(g, adj, rows, dev)
    n, cap_n, ex = h["n"], h["cap_n"], h["ex"]
    deg = torch.from_numpy(adj.indptr[1:] - adj.indptr[:-1])
    affected = (deg[rows] == 0) & torch.isin(rows, h["batch"])
    assert int(affected.sum()) > 0, "the hop has no expanded frontier row without out-edges"
    e_src = h["src_ref"].to(dev, torch.int32)
    e_dst = h["dst_ref"].to(dev, torch.int32)
    dl = torch.randn(cap_n, generator=torch.Generator().manual_seed(3))
    dl_d = dl.to(dev)
    dz = torch.full((cap_n,), NAN, device=dev)
    _L().grapes_aggregate_scalar_T(g.ctx, _p(dl_d), _p(h["n_dev"]), cap_n, _p(ex["P"]), 256, _p(ex["row_off"]),
                                   _p(e_src), _p(e_dst), _p(h["dinv"]),
                                   _p(ex["bm_rows"]) if fused else None, _p(h["batch_nodes"]) if fused else None,
                                   _p(g.indptr) if fused else None, _p(dz), _st())
    torch.cuda.synchronize()
    dinv = h["dinv_ref"]
    s, t = h["src_ref"], h["dst_ref"]
    keep = s != t
    s, t = s[keep], t[keep]
    dl64 = dl[:n].double()
    ref = (dinv * dinv * dl64).index_add(0, s, dinv[s] * dinv[t] * dl64[t])
    got = dz[:n].cpu()
    unwritten = torch.isnan(got).nonzero().squeeze(1).tolist()
    assert not unwritten, f"dz rows never written: {unwritten[:10]}"
    assert _rel(got, ref) < TOL, "dz differs from float64 A_hat^T dl"
    assert bool(torch.isnan(dz[n:]).all()), "written past n"


def test_aggregate_scalar_T_forms_agree_bit_for_bit(cuda_device, graph):
    """The fused form equals the two-launch form bit for bit (the same expression per row)."""
    d, adj, g = graph
    dev = cuda_device
    h = _hop_csr(g, adj, _rows(d, adj), dev)
    ex, cap_n = h["ex"], h["cap_n"]
    e_src, e_dst = h["src_ref"].to(dev, torch.int32), h["dst_ref"].to(dev, torch.int32)
    dl = torch.randn(cap_n, generator=torch.Generator().manual_seed(4)).to(dev)
    out = []
    for fused in (True, False):
        dz = torch.full((cap_n,), NAN, device=dev)
        _L().grapes_aggregate_scalar_T(g.ctx, _p(dl), _p(h["n_dev"]), cap_n, _p(ex["P"]), 256, _p(ex["row_off"]),
                                       _p(e_src), _p(e_dst), _p(h["dinv"]),
                                       _p(ex["bm_rows"]) if fused else None, _p(h["batch_nodes"]) if fused else None,
                                       _p(g.indptr) if fused else None, _p(dz), _st())
        out.append(dz)
    torch.cuda.synchronize()
    n = h["n"]
    assert torch.equal(out[0][:n], out[1][:n])


# ---- sampler net layer 1, SIMT form (main.py:112-114): z = relu(Y W1^T + b1) . w2 and its backward ----------------------
@pytest.fixture(scope="module")
def big_ctx(cuda_device):
    """a context whose split-K partial buffer holds what grapes_sampler_l1_bwd needs at D = 384, K = 1433"""
    from grapes_b200.graph import DeviceGraph
    return DeviceGraph(torch.zeros(2, dtype=torch.int64, device=cuda_device),
                       torch.zeros(0, dtype=torch.int32, device=cuda_device), 1, max_frontier=1 << 20,
                       partials_bytes=256 << 20)


def _sampler_inputs(K, D, n, cap_n, seed):
    """Y [cap_n, ldy] (finite junk in rows past n and in the pitch padding), W1 [D, K], b1, w2.  The kernels export no
    relu mask, so a pre-activation whose sign fp32 rounding could flip would make the float64 comparison meaningless:
    rows of Y are redrawn until every float64 |pre| over the n live rows is at least 1e-4 of the largest."""
    gen = torch.Generator().manual_seed(seed)
    ldy = (K + 3) // 4 * 4
    Y = torch.randn(cap_n, ldy, generator=gen)
    W1 = torch.randn(D, K, generator=gen) / K ** 0.5
    b1 = torch.randn(D, generator=gen) * 0.1
    w2 = torch.randn(D, generator=gen) / D ** 0.5
    for _ in range(100):
        pre = Y[:n, :K].double() @ W1.double().t() + b1.double()
        near = (pre.abs() < 1e-4 * pre.abs().max()).any(1)
        if not bool(near.any()):
            break
        Y[:n][near] = torch.randn(int(near.sum()), ldy, generator=gen)
    assert not bool(near.any())
    return Y, ldy, W1, b1, w2, pre


@pytest.mark.parametrize("K", [15, 41, 1433])
@pytest.mark.parametrize("D", [128, 256, 384])
def test_sampler_l1_simt(cuda_device, big_ctx, K, D):
    """Forward z and, with scale != 1 and accumulate = 1 onto nonzero gradients, the backward (dpre, gW1, gb1, gw2)
    against float64, for K not a multiple of 4 or 16 and n = 1000 (not a multiple of the 128-row tile)."""
    dev, L, ctx = cuda_device, _L(), big_ctx.ctx
    n, cap_n = 1000, 1100
    Y, ldy, W1, b1, w2, pre = _sampler_inputs(K, D, n, cap_n, K * 1000 + D)
    Yd, W1d, b1d, w2d = Y.to(dev), W1.to(dev), b1.to(dev), w2.to(dev)
    n_dev = _i32(n, dev)
    z = torch.full((cap_n,), NAN, device=dev)
    L.grapes_sampler_l1_fwd(ctx, _p(Yd), ldy, _p(n_dev), cap_n, K, _p(W1d), K, D, _p(b1d), _p(w2d), _p(z), _st())
    h64 = pre.clamp_min(0)
    assert _rel(z[:n], h64 @ w2.double()) < TOL, "z"
    assert bool(torch.isnan(z[n:]).all()), "z written past n"

    gen = torch.Generator().manual_seed(D)
    dz = torch.randn(cap_n, generator=gen)
    dpre64 = dz[:n].double().unsqueeze(1) * w2.double() * (pre > 0)
    grads = {"gW1": dpre64.t() @ Y[:n, :K].double(), "gb1": dpre64.sum(0), "gw2": h64.t() @ dz[:n].double()}
    init = {k: torch.randn(v.shape, generator=gen, dtype=torch.float64) * v.abs().max() for k, v in grads.items()}
    got = {k: v.float().to(dev) for k, v in init.items()}
    dzd = dz.to(dev)
    dpre = torch.full((cap_n, D), NAN, device=dev)
    scale = 0.37
    L.grapes_sampler_l1_bwd(ctx, _p(Yd), ldy, _p(n_dev), cap_n, K, _p(W1d), K, D, _p(b1d), _p(w2d), _p(dzd), _p(dpre),
                            scale, 1, _p(got["gW1"]), K, _p(got["gb1"]), _p(got["gw2"]), _st())
    torch.cuda.synchronize()
    assert _rel(dpre[:n], dpre64) < TOL, "dpre"
    for k in grads:
        assert _rel(got[k], init[k].float().double() + scale * grads[k]) < TOL, k


# ---- one hop of the sampler head, frontier mode: width-1 aggregation -> logits, then the selection -------------------
_NOISE = {"gumbel": 1, "keys": 3, "topk_probs": 4}


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


@pytest.mark.parametrize("nparts", [1, 4])
@pytest.mark.parametrize("mode,k", [("gumbel", 64), ("keys", 64), ("topk_probs", 64), ("gumbel", 100_000)])
def test_select_hop_frontier(cuda_device, graph, nparts, mode, k):
    """logits_all of every frontier row against float64 of the width-1 aggregation (nparts partial vectors summed on the
    fly; 4 = 2 D / 128 at D = 256); then every selection output bit for bit equal to grapes_select_topk fed the kernel's own
    candidate logits: sampled ids behind sampled_offset, s / total, keys, mask, log_prob, tot_log_prob, the min / max
    probability, sum_dl, bm_mark, and dl_all scattered to the candidates' frontier rows with 0 on every other row; the
    entropy mean / std against float64.  k = 100000 >= c is the take-all branch."""
    d, adj, g = graph
    dev, L = cuda_device, _L()
    h = _hop_csr(g, adj, _rows(d, adj), dev)
    n, cap_n, W = h["n"], h["cap_n"], g.num_words
    c = h["nb"].numel()
    assert 64 < c < n
    gen = torch.Generator().manual_seed(nparts * 7 + k)
    z = torch.randn(nparts, cap_n, generator=gen)
    zd = z.to(dev)
    bias = torch.tensor([-0.25], device=dev)
    nb_index = torch.cat([h["nb_index"], torch.full((cap_n - n,), -1, dtype=torch.int64)]).to(dev, torch.int32)
    nb_local = torch.cat([h["nb_local"], torch.zeros(cap_n - c, dtype=torch.int64)]).to(dev, torch.int32)
    nb_nodes = torch.cat([h["nb"], torch.zeros(cap_n - c, dtype=torch.int64)]).to(dev, torch.int32)
    c_dev = _i32(c, dev)
    offset = 5

    def outputs(cap):
        o = dict(keys=torch.full((cap,), NAN, device=dev), sampled=torch.full((offset + cap,), -1, dtype=torch.int32,
                 device=dev), s=_i32(-1, dev), total=_i32(-1, dev),
                 mask=torch.full((cap,), 0xAB, dtype=torch.uint8, device=dev), log_prob=torch.full((cap,), NAN, device=dev),
                 tot=torch.zeros(1, device=dev), stats=torch.zeros(4, device=dev), sum_dl=torch.zeros(1, device=dev),
                 bm=torch.zeros(W, dtype=torch.int32, device=dev), ukeys=torch.empty(cap, dtype=torch.int32, device=dev),
                 work=torch.zeros(int(L.cdll.grapes_select_work_floats(g.ctx, cap)), device=dev))
        assert o["work"].data_ptr() % 16 == 0
        return o

    ref_logits = _agg_ref(z.double().sum(0), h["off_ref"], h["val_ref"], h["dinv_ref"], -0.25)
    noise = None
    if mode != "topk_probs":
        noise = rp.draw_gumbel_like_reference(c, gen)
        if mode == "keys":
            noise = rp.perturbed_keys(ref_logits[h["nb_local"]].float(), noise)
        noise = noise.float().to(dev)
    hop = outputs(cap_n)
    logits_all = torch.full((cap_n,), NAN, device=dev)
    dl_all = torch.full((cap_n,), NAN, device=dev)
    L.grapes_select_hop(g.ctx, _p(zd), nparts, cap_n, _p(h["n_dev"]), cap_n, _p(h["in_off"]), _p(h["in_src"]),
                        _p(h["dinv"]), _p(bias), _p(nb_index), _p(nb_local), _p(nb_nodes), _p(c_dev), k, _NOISE[mode],
                        _p(noise), None, _p(hop["work"]), _p(hop["ukeys"]), _p(logits_all), _p(hop["keys"]),
                        _p(hop["sampled"]), offset, _p(hop["s"]), _p(hop["total"]), _p(hop["mask"]), _p(hop["log_prob"]),
                        _p(hop["tot"]), _p(hop["stats"]), _p(dl_all), _p(hop["sum_dl"]), _p(hop["bm"]), _st())
    torch.cuda.synchronize()
    assert _rel(logits_all[:n], ref_logits) < TOL, "logits_all"
    cand = logits_all[nb_local[:c].long()].clone()
    cap_c = c + 19
    lg = torch.cat([cand, torch.full((cap_c - c,), 3.5, device=dev)])
    top = outputs(cap_c)
    dl_c = torch.full((cap_c,), NAN, device=dev)
    L.grapes_select_topk(g.ctx, _p(lg), None, _p(nb_nodes), _p(c_dev), cap_c, k, _NOISE[mode], _p(noise), None,
                         _p(top["ukeys"]), _p(top["work"]), _p(top["keys"]), _p(top["sampled"]), offset, _p(top["s"]),
                         _p(top["total"]), _p(top["mask"]), _p(top["log_prob"]), _p(top["tot"]), _p(top["stats"]),
                         _p(dl_c), _p(top["sum_dl"]), _p(top["bm"]), _st())
    torch.cuda.synchronize()
    s = int(hop["s"].item())
    assert s == min(k, c) and int(hop["total"].item()) == offset + s
    for key in ("s", "total", "tot", "sum_dl", "bm"):
        assert torch.equal(_bits(hop[key]), _bits(top[key])), key
    if k >= c:
        assert torch.equal(_bits(hop["stats"]), _bits(top["stats"])), "stats"       # zero: the reference returns {}
    else:
        # min / max probability bit for bit; the entropy mean / std are fp32 sums whose split across threads follows the
        # rows each launch walks (frontier rows here, candidates there), so they hold the float64 bar of the selection
        # tests' statistics (1e-4: the std comes from the difference of two sums)
        assert torch.equal(_bits(hop["stats"][:2]), _bits(top["stats"][:2])), "stats: min / max probability"
        p64 = torch.sigmoid(cand.double().cpu())
        ent = -(p64 * torch.log2(p64) + (1 - p64) * torch.log2(1 - p64))
        for i, v in ((2, ent.mean()), (3, ent.std())):
            assert abs(hop["stats"][i].item() - v.item()) <= 1e-4 * abs(v.item()), f"stats[{i}] against float64"
            assert abs(top["stats"][i].item() - v.item()) <= 1e-4 * abs(v.item()), f"stats[{i}] of select_topk"
    assert torch.equal(hop["sampled"][:offset + s], top["sampled"][:offset + s]), "sampled"
    for key in ("keys", "mask", "log_prob"):
        assert torch.equal(_bits(hop[key][:c]), _bits(top[key][:c])), key
    want_dl = torch.zeros(n, device=dev)
    want_dl[nb_local[:c].long()] = dl_c[:c]
    assert torch.equal(_bits(dl_all[:n]), _bits(want_dl)), "dl_all"
