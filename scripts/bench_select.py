"""Micro-benchmark of the selection head on products- / Reddit-sized candidate sets (k = 256): CUDA-event time of
grapes_select_topk (k_select_fused, one launch on every SM) with its in-kernel phase stamps."""
import ctypes, os, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from grapes_b200._lib import lib, ptr
from grapes_b200.utils import _any_ctx

def main():
    dev = torch.device("cuda", 0)
    L = lib(); ctx = _any_ctx(dev).ctx
    for c in (8192, 65536, 150000):
        k = 256
        logits = torch.randn(c, device=dev) * 2
        nb = torch.arange(c, device=dev, dtype=torch.int32)
        cnt = torch.tensor([c, 0, 0, 0], dtype=torch.int32, device=dev)
        ukeys = torch.empty(c, dtype=torch.int32, device=dev)
        work = torch.zeros(int(L.cdll.grapes_select_work_floats(ctx, c)), dtype=torch.float32, device=dev)
        sampled = torch.empty(c, dtype=torch.int32, device=dev)
        lp = torch.empty(c, device=dev); dl = torch.empty(c, device=dev)
        stats = torch.zeros(4, device=dev); acc = torch.zeros(2, device=dev)
        rng = torch.tensor([1, 0], dtype=torch.int64, device=dev)
        st = torch.cuda.current_stream().cuda_stream
        def run():
            L.grapes_select_topk(ctx, ptr(logits), None, ptr(nb), cnt.data_ptr(), c, k, 0, None, ptr(rng), ptr(ukeys),
                                 ptr(work), None, ptr(sampled), 0, cnt.data_ptr() + 4, None, None, ptr(lp),
                                 acc.data_ptr(), ptr(stats), ptr(dl), acc.data_ptr() + 4, None, st)
        for _ in range(5): run()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda._sleep(2_000_000)
        e0.record()
        for _ in range(20): run()
        e1.record(); torch.cuda.synchronize()
        o8 = (ctypes.c_int64 * 8)()
        L.cdll.grapes_debug_select_fused_stamps(ctx, ctypes.c_void_p(work.data_ptr()), c, o8)
        t8 = list(o8)
        n8 = ["start", "keys done", "hist merged", "barrier 1", "members listed", "barrier 2", "outputs done", "last block done"]
        rel = {n8[i]: round((t8[i] - t8[0]) / 1e3, 2) for i in range(8)}
        print(f"c={c}: {e0.elapsed_time(e1) / 20 * 1e3:.1f} us per select; stamps us: {rel}")

if __name__ == "__main__":
    main()
