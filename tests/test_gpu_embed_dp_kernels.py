"""The kernels of the data-parallel learned table on ONE GPU: grapes_embed_merge_adam on hand-built slots of several ranks
(union, rank-order mean rows, dense Adam) and grapes_step_tail_embed with a world of one (payload pushed into its own
second buffer under the step's flag, merged through the go word; a failed exchange is a no-op)."""
import ctypes

import pytest
import torch

from test_gpu_embed import _bitmap

pytestmark = pytest.mark.gpu


def _ctx(N, dev):
    from grapes_b200.graph import DeviceGraph
    gen = torch.Generator().manual_seed(1)
    return DeviceGraph.from_edge_index(torch.randint(0, N, (2, 4 * N), generator=gen), N, device=dev)


def _slots(payloads, cap, F):
    from grapes_b200._lib import lib
    slot = int(lib().cdll.grapes_embed_slot_floats(cap, F))
    buf = torch.zeros(len(payloads) * slot, dtype=torch.float32)
    cap4 = (cap + 3) // 4 * 4
    for r, (ids, rows) in enumerate(payloads):
        s = buf[r * slot:(r + 1) * slot]
        s.view(torch.int32)[0] = ids.numel()
        s.view(torch.int32)[4:4 + ids.numel()] = ids.to(torch.int32)
        s[4 + cap4:4 + cap4 + rows.numel()] = rows.reshape(-1)
    return buf, slot


def _merge_args(N, F, cap_U, dev):
    W = (N + 31) // 32
    i32 = dict(dtype=torch.int32, device=dev)
    return dict(bm=torch.zeros(W, **i32), pref=torch.zeros(W + 1, **i32), ids=torch.zeros(cap_U, **i32),
                cnt=torch.zeros(1, **i32), mean=torch.zeros(cap_U, F, device=dev), ovf=torch.zeros(1, **i32))


def _merge(L, g, slots, world, cap, F, state, a, tab, m, v, N, lr, steps):
    L.grapes_embed_merge_adam(g.ctx, slots.data_ptr(), world, cap, F, state, a["bm"].data_ptr(), a["pref"].data_ptr(),
                              a["ids"].data_ptr(), a["ids"].numel(), a["cnt"].data_ptr(), a["mean"].data_ptr(),
                              tab.data_ptr(), m.data_ptr(), v.data_ptr(), N, lr, 0.9, 0.999, 1e-8, steps.data_ptr(),
                              a["ovf"].data_ptr(), torch.cuda.current_stream().cuda_stream)


def test_merge_of_three_ranks_matches_mean_gradient_and_dense_adam(cuda_device):
    from grapes_b200._lib import lib
    dev, L = cuda_device, lib()
    N, F, cap, world, lr = 1000, 16, 96, 3, 1e-2
    g = _ctx(N, dev)
    gen = torch.Generator().manual_seed(7)
    x = torch.randn(N, F, generator=gen)
    ref = torch.nn.Parameter(x.clone().double())
    opt = torch.optim.Adam([ref], lr=lr)
    tab, m, v = x.to(dev), torch.zeros(N, F, device=dev), torch.zeros(N, F, device=dev)
    steps = torch.zeros(2, device=dev)
    for it in range(3):
        payloads = []
        for r in range(world):
            ids = torch.sort(torch.randperm(N, generator=gen)[:int(torch.randint(1, cap + 1, (1,), generator=gen))]).values
            payloads.append((ids, torch.randn(ids.numel(), F, generator=gen)))
        slots, _ = _slots(payloads, cap, F)
        slots = slots.to(dev)
        a = _merge_args(N, F, world * cap, dev)
        steps[0] += 1                                  # the parameter Adam of the step ran first
        _merge(L, g, slots, world, cap, F, None, a, tab, m, v, N, lr, steps)
        dense = torch.zeros(N, F)
        for ids, rows in payloads:                     # rank order, fp32, like the kernel
            dense[ids] = dense[ids] + rows
        dense = dense * (1.0 / world)
        union = torch.unique(torch.cat([p[0] for p in payloads]))
        U = int(a["cnt"].item())
        assert torch.equal(a["ids"][:U].cpu().long(), union)
        assert torch.equal(a["mean"][:U].cpu(), dense[union])
        opt.zero_grad()
        ref.grad = dense.double()
        opt.step()
        assert (tab.double().cpu() - ref.detach()).abs().max() < 2e-6 * (it + 1)
    assert int(a["ovf"].item()) == 0


def test_tail_embed_world_one_equals_single_gpu_update_and_failure_is_a_noop(cuda_device):
    from grapes_b200._lib import lib
    dev, L = cuda_device, lib()
    N, F, cap, n, lr = 1000, 16, 64, 3000, 1e-3
    g = _ctx(N, dev)
    gen = torch.Generator().manual_seed(3)
    st_ = torch.cuda.current_stream().cuda_stream
    f32 = dict(dtype=torch.float32, device=dev)
    params, m_p, v_p = torch.randn(n, generator=gen).to(dev), torch.zeros(n, **f32), torch.zeros(n, **f32)
    x = torch.randn(N, F, generator=gen).to(dev)
    tab, m, v = x.clone(), torch.zeros(N, F, **f32), torch.zeros(N, F, **f32)
    tab1, m1, v1 = x.clone(), torch.zeros(N, F, **f32), torch.zeros(N, F, **f32)      # single-GPU path
    steps, steps1 = torch.zeros(2, **f32), torch.zeros(2, **f32)
    pbuf = torch.zeros(int(L.cdll.grapes_peer_buffer_floats(n, 1)), **f32)
    ebuf = torch.zeros(int(L.cdll.grapes_embed_peer_buffer_floats(cap, F, 1)), **f32)
    peers, epeers = (ctypes.c_void_p * 1)(pbuf.data_ptr()), (ctypes.c_void_p * 1)(ebuf.data_ptr())
    state = torch.zeros(int(L.cdll.grapes_peer_state_words()), dtype=torch.int32, device=dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    a = _merge_args(N, F, cap, dev)

    def step(grads, ids, rows):
        A = torch.tensor([ids.numel()], dtype=torch.int32, device=dev)
        ids_d = torch.zeros(cap, dtype=torch.int32, device=dev)
        ids_d[:ids.numel()] = ids.to(dev, torch.int32)
        rows_d = torch.zeros(cap, F, **f32)
        rows_d[:ids.numel()] = rows.to(dev)
        L.grapes_step_tail_embed(g.ctx, None, 0, 0.0, 0.0, 0, 0, None, 0, 0, 0, 0, peers, epeers, 0, 1, n,
                                 params.data_ptr(), grads.data_ptr(), m_p.data_ptr(), v_p.data_ptr(), 0, n, lr, 0, 0,
                                 1e-4, 0.9, 0.999, 1e-8, steps.data_ptr(), state.data_ptr(), err.data_ptr(),
                                 A.data_ptr(), ids_d.data_ptr(), rows_d.data_ptr(), F, F, cap, st_)
        a["bm"].zero_()
        _merge(L, g, ebuf, 1, cap, F, state.data_ptr(), a, tab, m, v, N, lr, steps)
        return A, ids_d, rows_d

    for it in range(4):
        ids = torch.sort(torch.randperm(N, generator=gen)[:10 + 15 * it]).values
        rows = torch.randn(ids.numel(), F, generator=gen)
        grads = torch.randn(n, generator=gen).to(dev)
        step(grads, ids, rows)
        bm1, pref1 = _bitmap(ids, N, dev)
        L.grapes_adam_embed(g.ctx, tab1.data_ptr(), m1.data_ptr(), v1.data_ptr(), N, F, bm1.data_ptr(), pref1.data_ptr(),
                            rows.to(dev).data_ptr(), F, lr, 0.9, 0.999, 1e-8, steps1.data_ptr(), st_)
        steps1[0] += 1
        torch.cuda.synchronize()
        assert int(err.item()) == 0 and int(state[0].item()) == it + 1
        slot = ebuf[(it + 1) % 2 * ebuf.numel() // 2:]                 # parity of step it + 1
        assert int(slot.view(torch.int32)[0].item()) == ids.numel()
        assert torch.equal(slot.view(torch.int32)[4:4 + ids.numel()].cpu(), ids.to(torch.int32))
        assert torch.equal(a["ids"][:int(a["cnt"].item())].cpu().long(), ids)
        for got, want in ((tab, tab1), (m, m1), (v, v1)):              # W = 1: exactly the single-GPU table step
            assert torch.equal(got, want)
        assert float(steps[0]) == it + 1
    # a failed exchange (sticky failure word): flagged, table / moments / parameters / step counts untouched
    state[3] = 1
    before = [t.clone() for t in (tab, m, v, params, m_p, v_p, steps)]
    step(torch.randn(n, generator=gen).to(dev), torch.arange(5), torch.randn(5, F, generator=gen))
    torch.cuda.synchronize()
    assert int(err.item()) & 32
    for b, t in zip(before, (tab, m, v, params, m_p, v_p, steps)):
        assert torch.equal(b, t)
