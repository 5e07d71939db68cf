"""Directed variants of make_synth's graphs, shared by the directed-graph tests (test_gpu_directed.py) and the hop-kernel
tests (test_gpu_hop_kernels.py).  make_synth emits both directions of every pair, so its graphs are their own transpose;
these are not, and they hold expanded rows without out-edges that other rows point to."""
import torch


def directed_synth(name, seed, power_law=0.0):
    """make_synth's data with a directed graph: each pair of synth_edge_index kept in ONE random direction, every
    out-edge of a random fifth of the nodes dropped, then a few stored self-loops and duplicated edges added."""
    from grapes_b200.synth import make_synth
    d = make_synth(name, seed=seed, power_law=power_law)
    N = d.num_nodes
    g = torch.Generator().manual_seed(10_000 + seed)
    half = d.edge_index.shape[1] // 2
    pairs = d.edge_index[:, :half]                            # synth_edge_index: [pairs, pairs.flip(0)]
    flip = torch.rand(half, generator=g) < 0.5
    pairs = torch.where(flip, pairs.flip(0), pairs)
    sink = torch.zeros(N, dtype=torch.bool)
    sink[torch.randperm(N, generator=g)[:N // 5]] = True
    pairs = pairs[:, ~sink[pairs[0]]]
    loops = torch.randint(0, N, (8,), generator=g).repeat(2, 1)
    dups = pairs[:, torch.randint(0, pairs.shape[1], (16,), generator=g)]
    d.edge_index = torch.cat([pairs, loops, dups], dim=1)
    return d


def empty_expanded_frontier_rows(adjacency, prev, batch_nodes) -> int:
    """rows of a hop that are expanded AND frontier nodes while having no out-edge"""
    deg = torch.from_numpy(adjacency.indptr[1:] - adjacency.indptr[:-1])
    prev = prev.cpu().long()
    return int(((deg[prev] == 0) & torch.isin(prev, batch_nodes.cpu().long())).sum())
