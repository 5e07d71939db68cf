"""CPU tests of the data-parallel evaluation's host logic: the row partition of the full-batch forward (a numpy mirror of
``grapes_graph_norm_window_bounds``, which the GPU tests compare the kernel against), the mini-batch assignment, and the
integer count reduction and prediction reassembly in a world-size-2 gloo run."""
import os
import socket

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from grapes_b200.dist import allreduce_counts_, eval_batches, gather_batch_predictions


def row_partition(in_off, world: int):
    """bounds[k] = the least i in [0, N] with (in_off[i] + i) * W >= k * (in_off[N] + N), k = 0 .. W."""
    in_off = np.asarray(in_off, dtype=np.int64)
    N = in_off.shape[0] - 1
    prefix = (in_off + np.arange(N + 1, dtype=np.int64)) * world
    T = int(in_off[-1]) + N
    return [int(np.searchsorted(prefix, k * T, side="left")) for k in range(world + 1)]


def _in_off(indeg):
    return np.concatenate([[0], np.cumsum(indeg)]).astype(np.int64)


def test_partition_is_contiguous_and_balanced():
    rng = np.random.default_rng(0)
    cases = [rng.integers(0, 50, 1000), rng.zipf(1.6, 3000).clip(max=100_000), np.zeros(17, dtype=np.int64),
             np.array([5]), np.array([0, 0, 9]), np.array([100_000, 1, 1, 1, 1, 1, 1, 1, 1, 1])]
    for indeg in cases:
        in_off = _in_off(indeg)
        N = len(indeg)
        weight = indeg + 1
        for W in (1, 2, 3, 4, 7, 8):
            b = row_partition(in_off, W)
            assert b == row_partition(in_off.copy(), W)                  # deterministic
            assert b[0] == 0 and b[-1] == N and all(b[k] <= b[k + 1] for k in range(W))
            total = int(weight.sum())
            heaviest = int(weight.max())
            for k in range(W):
                load = int(weight[b[k]:b[k + 1]].sum())
                assert abs(load - total / W) <= heaviest, (W, k, load, total / W)


def test_partition_leaves_windows_empty_when_there_are_fewer_rows_than_ranks():
    b = row_partition(_in_off(np.array([2, 0, 1])), 8)
    assert b[0] == 0 and b[-1] == 3
    sizes = [b[k + 1] - b[k] for k in range(8)]
    assert sum(sizes) == 3 and sizes.count(0) == 5 and max(sizes) == 1


def test_eval_batches_cover_every_batch_once_tail_included():
    for nb, world in ((10, 2), (11, 4), (3, 8), (0, 2), (105, 8), (1, 1)):
        shards = [eval_batches(nb, r, world) for r in range(world)]
        assert sorted(i for s in shards for i in s) == list(range(nb))
        for r, s in enumerate(shards):
            assert all(i % world == r for i in s) and s == sorted(s)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(1)
    sizes = [4, 4, 4, 4, 4, 2]                                          # tail batch of 2, odd number of batches
    truth = torch.arange(sum(sizes), dtype=torch.int64) * 3 + 1
    starts = np.concatenate([[0], np.cumsum(sizes)])
    mine = eval_batches(len(sizes), rank, world)
    local = torch.cat([truth[starts[i]:starts[i + 1]] for i in mine])
    counts = torch.tensor([rank + 1, 10 * (rank + 1), 0], dtype=torch.int64)
    allreduce_counts_(counts)
    preds = gather_batch_predictions(local, sizes)
    one = gather_batch_predictions(truth[:3] if rank == 0 else truth[:0], [3])    # more ranks than batches
    out[rank] = dict(preds=preds, counts=counts.clone(), truth=truth, one=one)
    dist.barrier()
    dist.destroy_process_group()


def test_count_reduction_and_prediction_reassembly_gloo():
    world = 2
    out = mp.Manager().dict()
    mp.spawn(_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    for r in range(world):
        got = out[r]
        assert torch.equal(got["preds"], got["truth"])
        assert got["counts"].tolist() == [3, 30, 0]
        assert torch.equal(got["one"], got["truth"][:3])
