"""GCNConv / GCN parity (SURVEY.md section 8 rows a6, a7, a11, a12): logits and gradients within
1e-5 relative (to the tensor's scale) of the fp64 restatement of PyG 2.5.2 GCNConv."""
import pytest
import torch

from oracle import reference_port as rp

pytestmark = pytest.mark.gpu
TOL = 1e-5


def _close(got, ref, tol=TOL):
    ref = ref.double()
    scale = ref.abs().max().clamp_min(1e-30)
    err = (got.double().cpu() - ref).abs().max() / scale
    assert err < tol, f"relative error {err:.3e} >= {tol}"


def _rand_graph(n, E, gen):
    ei = torch.randint(0, n, (2, E), generator=gen)
    return ei


@pytest.mark.parametrize("n,E,dims", [(50, 200, [12, 32, 5]), (1661, 2071, [104, 256, 1]),
                                     (544, 700, [100, 256, 47]), (300, 5000, [33, 17, 3])])
def test_gcn_forward_backward(cuda_device, n, E, dims):
    from grapes_b200.gcn import GCN
    gen = torch.Generator().manual_seed(n)
    ei = _rand_graph(n, E, gen)
    ei[:, :5] = ei[0, :5]                    # a few explicit self-loops (must be replaced, not doubled)
    x = torch.randn(n, dims[0], generator=gen)
    ref = rp.OracleGCN(dims[0], dims[1:], generator=gen).double()
    net = GCN(dims[0], dims[1:]).to(cuda_device)
    net.load_state_dict({k: v.float() for k, v in ref.state_dict().items()})
    out_ref, _ = ref(x.double(), ei)
    w = torch.randn(out_ref.shape, generator=gen).double()
    (out_ref * w).sum().backward()
    out, mem = net(x.to(cuda_device), ei.to(cuda_device))
    assert isinstance(mem, float)
    (out * w.float().to(cuda_device)).sum().backward()
    _close(out, out_ref.detach())
    for (name, p), (_, pr) in zip(net.named_parameters(), ref.named_parameters()):
        _close(p.grad, pr.grad)


def test_gcn_layerwise_edge_list_quirk(cuda_device):
    """With a list of 3 blocks the hidden layer uses edges[-1] and the last layer edges[0]; edges[1] is
    never consumed (gcn.py:30-36, SURVEY.md section 3.1 'layer-index quirk')."""
    from grapes_b200.gcn import GCN
    gen = torch.Generator().manual_seed(0)
    n = 200
    edges = [_rand_graph(n, 300, gen) for _ in range(3)]
    x = torch.randn(n, 20, generator=gen)
    ref = rp.OracleGCN(20, [64, 7], generator=gen).double()
    net = GCN(20, [64, 7]).to(cuda_device)
    net.load_state_dict({k: v.float() for k, v in ref.state_dict().items()})
    out_ref, _ = ref(x.double(), edges)
    out, _ = net(x.to(cuda_device), [e.to(cuda_device) for e in edges])
    _close(out, out_ref.detach())
    edges2 = [edges[0], _rand_graph(n, 10, gen), edges[2]]
    out2, _ = net(x.to(cuda_device), [e.to(cuda_device) for e in edges2])
    assert torch.equal(out, out2)            # deterministic kernels: bitwise identical


def test_gcn_input_gradient(cuda_device):
    """dX path (needed by embed_nodes, SURVEY.md section 8 row f4)."""
    from grapes_b200.gcn import GCN
    gen = torch.Generator().manual_seed(3)
    n = 120
    ei = _rand_graph(n, 500, gen)
    x = torch.randn(n, 40, generator=gen)
    ref = rp.OracleGCN(40, [16, 4], generator=gen).double()
    net = GCN(40, [16, 4]).to(cuda_device)
    net.load_state_dict({k: v.float() for k, v in ref.state_dict().items()})
    xr = x.double().requires_grad_(True)
    ref(xr, ei)[0].square().sum().backward()
    xg = x.to(cuda_device).requires_grad_(True)
    net(xg, ei.to(cuda_device))[0].square().sum().backward()
    _close(xg.grad, xr.grad)


@pytest.mark.parametrize("F,num_ind,ones", [(100, 4, True), (36, 4, True), (100, 3, False), (64, 8, True), (256, 3, True)])
@pytest.mark.parametrize("hi_lo", [False, True])
def test_agg_tma_pad_columns_bit_identical_to_register_staged(cuda_device, F, num_ind, ones, hi_lo):
    """The TMA-staged aggregation with its pad columns (indicators | ones | zeros) == the register-staged kernel
    (grapes_agg_variant 1), bit for bit; the indicator columns equal the weighted sums of the source bits."""
    from grapes_b200._lib import lib, ptr
    from grapes_b200.graph import DeviceGraph
    dev = cuda_device
    gen = torch.Generator().manual_seed(F + num_ind)
    N, n = 30000, 9000
    g = DeviceGraph.from_edge_index(torch.randint(0, N, (2, 1000), generator=gen), N, device=dev)
    x = torch.randn(N, F, generator=gen).to(dev)
    nodes = torch.sort(torch.randperm(N, generator=gen)[:n]).values.to(torch.int32).to(dev)
    cnt_e = torch.randint(0, 6, (n,), generator=gen)
    cnt_e[5] = 300                                                     # one long row: several 16-entry chunks
    in_off = torch.zeros(n + 1, dtype=torch.int32)
    in_off[1:] = torch.cumsum(cnt_e, 0)
    in_src = torch.randint(0, n, (int(in_off[-1]),), generator=gen, dtype=torch.int32)
    dinv = (torch.rand(n, generator=gen) * 0.5 + 0.1).to(dev)
    bits = torch.randint(0, 1 << num_ind, (n,), generator=gen, dtype=torch.int32).to(dev)
    ldo = (F + num_ind + (1 if ones else 0) + 3) // 4 * 4
    ones_col = F + num_ind if ones else -1
    n_dev = torch.tensor([n], dtype=torch.int32, device=dev)
    in_off, in_src = in_off.to(dev), in_src.to(dev)
    L = lib()
    st = torch.cuda.current_stream().cuda_stream

    def run():
        a = torch.full((n, ldo), float("nan"), device=dev)
        b = torch.full((n, ldo), float("nan"), device=dev)
        L.grapes_aggregate(g.ctx, ptr(x), F, F, ptr(nodes), ptr(n_dev), n, ptr(in_off), ptr(in_src), ptr(dinv), ptr(bits),
                           num_ind, None, 0, None if hi_lo else ptr(a), ldo, ptr(a) if hi_lo else None,
                           ptr(b) if hi_lo else None, ones_col, st)
        torch.cuda.synchronize()
        return (a, b) if hi_lo else (a,)
    try:
        y_tma = run()
        L.cdll.grapes_agg_variant(1)
        y_reg = run()
    finally:
        L.cdll.grapes_agg_variant(0)
    for a, b in zip(y_tma, y_reg):
        assert not torch.isnan(a).any()
        assert torch.equal(a, b)
    y = y_tma[0] + y_tma[1] if hi_lo else y_tma[0]
    # reference of the pad columns in float64
    w_self = dinv.double() ** 2
    bitf = torch.stack([((bits >> i) & 1).double() for i in range(num_ind)], 1)
    ind = w_self[:, None] * bitf
    rows = torch.repeat_interleave(torch.arange(n, device=dev), cnt_e.to(dev))
    ind.index_add_(0, rows, (dinv.double()[in_src.long()] * dinv.double()[rows])[:, None] * bitf[in_src.long()])
    assert (y[:, F:F + num_ind].double() - ind).abs().max() < 1e-5 * ind.abs().max()
    if ones:
        assert bool((y[:, ones_col] == 1).all())
    assert bool((y[:, F + num_ind + (1 if ones else 0):] == 0).all())


@pytest.mark.parametrize("F,num_ind", [(602, 3), (1433, 3), (38, 4), (41, 0), (103, 4)])
@pytest.mark.parametrize("hi_lo", [False, True])
def test_agg_tma_width_not_multiple_of_4_bit_identical(cuda_device, F, num_ind, hi_lo):
    """Feature widths that are not a multiple of 4 floats (Reddit 602, Cora 1433) on a table with a padded row pitch: the
    TMA-staged aggregation (partial last feature lane) == the register-staged kernel, bit for bit; pad columns of the
    TABLE hold NaN canaries (they are staged and accumulated, never stored), every output column is written."""
    from grapes_b200._lib import lib, ptr
    from grapes_b200.graph import DeviceGraph
    dev = cuda_device
    gen = torch.Generator().manual_seed(F)
    N, n = 12000, 5000
    ldx = (F + 3) // 4 * 4
    g = DeviceGraph.from_edge_index(torch.randint(0, N, (2, 1000), generator=gen), N, device=dev)
    xp = torch.full((N, ldx), float("nan"))
    xp[:, :F] = torch.randn(N, F, generator=gen)
    xp = xp.to(dev)
    nodes = torch.sort(torch.randperm(N, generator=gen)[:n]).values.to(torch.int32).to(dev)
    cnt_e = torch.randint(0, 5, (n,), generator=gen)
    cnt_e[7] = 70
    in_off = torch.zeros(n + 1, dtype=torch.int32)
    in_off[1:] = torch.cumsum(cnt_e, 0)
    in_src = torch.randint(0, n, (int(in_off[-1]),), generator=gen, dtype=torch.int32).to(dev)
    in_off = in_off.to(dev)
    dinv = (torch.rand(n, generator=gen) * 0.5 + 0.1).to(dev)
    bits = torch.randint(0, 1 << max(num_ind, 1), (n,), generator=gen, dtype=torch.int32).to(dev)
    ones_col = F + num_ind
    ldo = (F + num_ind + 1 + 3) // 4 * 4
    n_dev = torch.tensor([n], dtype=torch.int32, device=dev)
    L = lib()
    st = torch.cuda.current_stream().cuda_stream

    def run():
        a = torch.full((n, ldo), float("nan"), device=dev)
        b = torch.full((n, ldo), float("nan"), device=dev)
        L.grapes_aggregate(g.ctx, ptr(xp), F, ldx, ptr(nodes), ptr(n_dev), n, ptr(in_off), ptr(in_src), ptr(dinv),
                           ptr(bits) if num_ind else None, num_ind, None, 0, None if hi_lo else ptr(a), ldo,
                           ptr(a) if hi_lo else None, ptr(b) if hi_lo else None, ones_col, st)
        torch.cuda.synchronize()
        return (a, b) if hi_lo else (a,)
    try:
        n0 = L.grapes_kernel_launches()
        y_tma = run()
        L.cdll.grapes_agg_variant(1)
        y_reg = run()
    finally:
        L.cdll.grapes_agg_variant(0)
    for a, b in zip(y_tma, y_reg):
        assert not torch.isnan(a).any() and torch.equal(a, b)
    y = (y_tma[0] + y_tma[1]) if hi_lo else y_tma[0]
    x = xp[:, :F].double()
    ref = (dinv.double() ** 2)[:, None] * x[nodes.long()]
    rows = torch.repeat_interleave(torch.arange(n, device=dev), cnt_e.to(dev))
    w = dinv.double()[in_src.long()] * dinv.double()[rows]
    ref.index_add_(0, rows, w[:, None] * x[nodes.long()[in_src.long()]])
    assert (y[:, :F].double() - ref).abs().max() < 1e-5 * ref.abs().max()
    assert bool((y[:, ones_col] == 1).all())
