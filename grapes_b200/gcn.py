"""Drop-in mirror of the reference's ``modules/gcn.py`` ``GCN`` (/root/reference/modules/gcn.py:9-42)
with ``torch_geometric.nn.GCNConv`` (PyG 2.5.2 defaults) replaced by the C-ABI CUDA kernels.

Parameter names follow PyG (``gcn_layers.{i}.lin.weight`` [out, in], ``gcn_layers.{i}.bias`` [out]) so a
reference ``state_dict`` loads unchanged.  ``forward`` returns ``(logits, memory_alloc_MB)`` like the
reference (gcn.py:40-42).
"""
from __future__ import annotations

import math
from typing import List, Union

import torch
import torch.nn as nn
import torch.nn.functional as F

from ._lib import lib, ptr, GrapesError
from .utils import _any_ctx, _stream


class NormAdj:
    """gcn_norm structure of one edge_index on n nodes: dst-sorted CSR (forward), src-sorted CSR
    (backward), deg^-1/2 with the added self-loops (SURVEY.md section 3.2 steps 1-3)."""

    def __init__(self, edge_index: torch.Tensor, n: int):
        if not edge_index.is_cuda:
            raise GrapesError("grapes_b200 has no CPU fallback: edge_index must live on a CUDA device")
        dev = edge_index.device
        self.holder = _any_ctx(dev)
        L, ctx = lib(), self.holder.ctx
        E = int(edge_index.shape[1])
        self.n, self.E = int(n), E
        src = edge_index[0].to(torch.int32).contiguous()
        dst = edge_index[1].to(torch.int32).contiguous()
        capE, capn = max(E, 1), max(self.n, 1)
        if max(capE, capn) > self.holder.max_frontier:
            raise GrapesError("edge list larger than the library context's max_frontier")
        self.cnt = torch.tensor([E, self.n, 0, 0, 0, 0], dtype=torch.int32, device=dev)
        scratch = torch.zeros(capn, dtype=torch.int32, device=dev)
        tmp = torch.empty(capE, dtype=torch.int32, device=dev)
        ovf = torch.zeros(1, dtype=torch.int32, device=dev)
        self.in_off = torch.zeros(capn + 1, dtype=torch.int32, device=dev)
        self.in_src = torch.empty(capE, dtype=torch.int32, device=dev)
        self.out_off = torch.zeros(capn + 1, dtype=torch.int32, device=dev)
        self.out_dst = torch.empty(capE, dtype=torch.int32, device=dev)
        self.dinv = torch.empty(capn, dtype=torch.float32, device=dev)
        c = self.cnt.data_ptr()
        L.grapes_build_csr(ctx, ptr(dst), ptr(src), c, capE, c + 4, capn, ptr(scratch), 0, ptr(self.in_off),
                           ptr(self.in_src), ptr(tmp), ptr(self.dinv), c + 8, ptr(ovf), _stream())
        L.grapes_build_csr(ctx, ptr(src), ptr(dst), c, capE, c + 4, capn, ptr(scratch), 0, ptr(self.out_off),
                           ptr(self.out_dst), ptr(tmp), None, c + 12, ptr(ovf), _stream())

    def aggregate(self, x: torch.Tensor, transpose: bool = False, bias=None) -> torch.Tensor:
        L, ctx = lib(), self.holder.ctx
        x = x.contiguous()
        Fdim = x.shape[1]
        out = torch.empty_like(x)
        off, idx = (self.out_off, self.out_dst) if transpose else (self.in_off, self.in_src)
        L.grapes_aggregate(ctx, ptr(x), Fdim, Fdim, None, self.cnt.data_ptr() + 4, max(self.n, 1), ptr(off), ptr(idx),
                           ptr(self.dinv), None, 0, ptr(bias), 0, ptr(out), Fdim, None, None, -1, _stream())
        return out


class GraphNorm(NormAdj):
    """gcn_norm structure of the WHOLE graph, built once from a :class:`DeviceGraph` (full-batch evaluation,
    /root/reference/eval.py:47-56: ``gcn_c(x, edge_index)`` over every edge).  PyG semantics (SURVEY.md 3.2):
    stored self-loops are dropped, one self-loop per node is added, deg = in-degree + 1; the in-neighbour lists are
    the CSR of the transposed adjacency (edge_index[0] = source row, edge_index[1] = destination column),
    ascending source inside a row.  Two builders of the same arrays (see ``__init__``): the default sorts the
    (destination, source) keys with ``torch.sort`` (one-off set-up); the opt-in "lib" builder uses the
    library's own kernels -- ``grapes_row_offsets`` + ``grapes_expand_rows`` turn the CSR back into its edge list,
    ``grapes_build_csr`` (counting sort by destination, per-row sort, self-loops dropped, deg^-1/2) is the routine that
    builds every hop's structure.  One-off, cached on the graph; the aggregation itself is ``grapes_aggregate``
    (TMA-staged SpMM) straight on these arrays.  nnz must fit int32 offsets; larger graphs use :class:`WideGraphNorm`."""

    def __init__(self, graph, edge_index=None, builder=None):
        """``builder``: "torch" (default) sorts the (destination, source) keys with
        ``torch.sort``; "lib" (``GRAPES_GRAPHNORM_BUILDER=lib``) builds the same arrays with the library's own kernels
        (``grapes_row_offsets`` / ``grapes_expand_rows`` / ``grapes_build_csr``), equal to the torch builder bit for bit
        (``tests/test_gpu_eval.py::test_lib_builder_equals_torch_builder``); it raises when ``grapes_build_csr`` flags an
        overflow.  ``bench.py --full-eval`` measures it in a process of its own."""
        import os
        builder = builder or os.environ.get("GRAPES_GRAPHNORM_BUILDER", "torch")
        self._own_ctx = None
        self.graph = graph
        self._edge_index = edge_index            # the transposed structure is built from the same input, on demand
        if builder == "lib":
            self._build_lib(graph, edge_index)
        else:
            self._build_torch(graph, edge_index)

    def _build_torch(self, graph, edge_index=None):
        """``edge_index`` given: the structure of THAT edge list (duplicates kept and counted, exactly what
        ``gcn_c(x, data.edge_index)`` sees in eval.py:50); otherwise the graph's canonical CSR (duplicates collapsed
        by main.py:134)."""
        dev = graph.device
        N = graph.num_nodes
        self.holder = graph
        if edge_index is not None:
            ei = edge_index.to(device=dev, dtype=torch.int64)
            src, dst = ei[0], ei[1]
        else:
            counts = graph.indptr[1:] - graph.indptr[:-1]
            src = torch.repeat_interleave(torch.arange(N, device=dev, dtype=torch.int64), counts)
            dst = graph.indices.to(torch.int64)
        if src.numel() >= (1 << 31) - 1:
            raise GrapesError("full-graph aggregation needs nnz < 2^31 per device")
        keep = src != dst
        key = dst[keep] * N + src[keep]
        del src, dst, keep
        self.n, self.E = N, int(key.numel())
        key = torch.sort(key).values
        d = torch.div(key, N, rounding_mode="floor")
        self.in_src = (key - d * N).to(torch.int32)
        del key
        indeg = torch.bincount(d, minlength=N)
        del d
        self.in_off = torch.zeros(N + 1, dtype=torch.int32, device=dev)
        self.in_off[1:] = torch.cumsum(indeg, 0).to(torch.int32)
        self.dinv = (1.0 / torch.sqrt((indeg + 1).to(torch.float32))).contiguous()
        self.cnt = torch.tensor([int(self.in_src.numel()), N, 0, 0, 0, 0], dtype=torch.int32, device=dev)
        self.out_off = self.out_dst = None

    def _build_lib(self, graph, edge_index=None):
        """``edge_index`` given: the structure of THAT edge list (duplicates kept and counted, exactly what
        ``gcn_c(x, data.edge_index)`` sees in eval.py:50); otherwise the graph's canonical CSR (duplicates collapsed
        by main.py:134)."""
        import ctypes
        dev = graph.device
        N = graph.num_nodes
        L = lib()
        st = _stream()
        E = int(edge_index.shape[1]) if edge_index is not None else graph.nnz
        if E >= (1 << 31) - 1:
            raise GrapesError("full-graph aggregation needs nnz < 2^31 per device")
        capE, capn = max(E, 1), max(N, 1)
        # a context whose scan scratch covers E entries (the graph's own is sized for frontiers)
        self._own_ctx = ctypes.c_void_p()
        rc = L.cdll.grapes_ctx_create(dev.index, N, max(capE, capn), 1 << 20, ctypes.byref(self._own_ctx))
        if rc != 0:
            raise GrapesError(f"grapes_ctx_create failed ({rc}): {L.last_error()}")
        ctx = self._own_ctx
        self.holder = self                       # NormAdj.aggregate reads holder.ctx
        self.graph = graph
        self.n, self.E = N, E
        cnt = torch.tensor([E, N, 0, 0, 0, 0], dtype=torch.int32, device=dev)
        c = cnt.data_ptr()
        if edge_index is not None:
            ei = edge_index.to(device=dev)
            src = ei[0].to(torch.int32).contiguous()
            dst = ei[1].to(torch.int32).contiguous()
        else:
            # the CSR back as an edge list: position of a row in `rows` == its id, so e_row is the source id
            rows = torch.arange(N, dtype=torch.int32, device=dev)
            row_off = torch.empty(N + 1, dtype=torch.int32, device=dev)
            src = torch.empty(capE, dtype=torch.int32, device=dev)
            dst = torch.empty(capE, dtype=torch.int32, device=dev)
            cntP = torch.tensor([N, 0, 0, 0], dtype=torch.int32, device=dev)
            L.grapes_row_offsets(ctx, ptr(graph.indptr), ptr(rows), cntP.data_ptr(), capn, ptr(row_off), cntP.data_ptr() + 4,
                                 capE, None, None, cntP.data_ptr() + 8, st)
            L.grapes_expand_rows(ctx, ptr(graph.indptr), ptr(graph.indices), ptr(rows), cntP.data_ptr(), capn, ptr(row_off),
                                 cntP.data_ptr() + 4, capE, ptr(src), ptr(dst), None, st)
            del rows, row_off
        scratch = torch.zeros(capn, dtype=torch.int32, device=dev)
        tmp = torch.empty(capE, dtype=torch.int32, device=dev)
        ovf = torch.zeros(1, dtype=torch.int32, device=dev)
        self.in_off = torch.zeros(capn + 1, dtype=torch.int32, device=dev)
        in_src = torch.empty(capE, dtype=torch.int32, device=dev)
        self.dinv = torch.empty(capn, dtype=torch.float32, device=dev)
        L.grapes_build_csr(ctx, ptr(dst), ptr(src), c, capE, c + 4, capn, ptr(scratch), 0, ptr(self.in_off), ptr(in_src),
                           ptr(tmp), ptr(self.dinv), c + 8, ptr(ovf), st)
        nnz = int(cnt[2].item())                 # stored entries without the dropped self-loops (one-off read-back)
        if int(ovf.item()) != 0:                 # e.g. more hub rows than the context's worklist holds: never a silent result
            raise GrapesError(f"GraphNorm (library builder): grapes_build_csr flagged overflow bits {int(ovf.item())}; "
                              "use builder='torch'")
        self.in_src = in_src[:nnz].clone() if nnz < capE else in_src
        del src, dst, tmp, scratch, in_src
        self.cnt = torch.tensor([nnz, N, 0, 0, 0, 0], dtype=torch.int32, device=dev)
        self.out_off = self.out_dst = None

    @property
    def ctx(self):
        return self._own_ctx if self._own_ctx is not None else self.graph.ctx

    def __del__(self):
        try:
            if getattr(self, "_own_ctx", None):
                lib().cdll.grapes_ctx_destroy(self._own_ctx)
                self._own_ctx = None
        except Exception:
            pass

    def aggregate(self, x, transpose=False, bias=None):
        """A_hat x (+ bias); ``transpose``: A_hat^T x (+ bias), the backward, on the transposed arrays built on the first
        call (:func:`transposed_structure`) with int32 offsets, through the same ``grapes_aggregate``."""
        if transpose:
            self.build_transposed()
        return super().aggregate(x, transpose, bias)

    def build_transposed(self):
        """The transposed arrays ``out_off`` (int32) / ``out_dst``, once."""
        if self.out_off is None:
            off, self.out_dst = transposed_structure(self.n, self.dinv.device, self.graph, self._edge_index)
            self.out_off = off.to(torch.int32)


class WideGraphNorm:
    """The same gcn_norm structure as :class:`GraphNorm` with int64 row offsets, for graphs of any edge count
    (``grapes_graph_norm_*``): ``in_off`` int64 [N+1], ``in_src`` int32 [nnz'], ``dinv`` fp32 [N], equal bit for bit to
    the torch-sort builder.  Built on the device by a counting sort by destination that reads the input where it lies:
    the graph's CSR, or ``edge_index`` (host or device, int64 [2, E]; duplicates kept and counted) in chunks of
    ``chunk_edges`` columns, so a host edge list never has to be on the device at once.  Without a graph (``graph=None``)
    the structure is that of ``edge_index`` on ``num_nodes`` nodes of ``device``.  Device memory beyond the outputs:
    ``grapes_graph_norm_workspace_bytes(N)`` (~4 N bytes) plus one chunk of a host edge list (16 bytes per edge).
    :meth:`aggregate_rows` aggregates one row slab (:func:`full_graph_forward_streamed`); :meth:`aggregate` all rows,
    forward or transposed (the backward of the drop-in module), the transposed arrays ``out_off`` / ``out_dst`` built
    from the same input on the first transposed call."""

    def __init__(self, graph, edge_index=None, chunk_edges: int = 1 << 27, *, num_nodes=None, device=None):
        if graph is None and (edge_index is None or num_nodes is None or device is None):
            raise GrapesError("WideGraphNorm without a graph needs edge_index, num_nodes and device")
        dev = graph.device if graph is not None else torch.device(device)
        N = graph.num_nodes if graph is not None else int(num_nodes)
        L, st = lib(), _stream()
        self.graph = graph
        self.holder = _any_ctx(dev)
        self._input = (edge_index, chunk_edges)
        self.out_off = self.out_dst = None
        self._slabs = None
        ws = torch.empty(max(int(L.cdll.grapes_graph_norm_workspace_bytes(N)), 1), dtype=torch.uint8, device=dev)
        err = torch.zeros(1, dtype=torch.int32, device=dev)
        nnz = torch.zeros(1, dtype=torch.int64, device=dev)
        self.in_off = torch.empty(N + 1, dtype=torch.int64, device=dev)
        self.dinv = torch.empty(N, dtype=torch.float32, device=dev)

        def run(pass_, in_src):
            if edge_index is None:
                L.grapes_graph_norm_add_csr(pass_, N, ptr(graph.indptr), ptr(graph.indices), 0, N, ptr(self.in_off),
                                            ptr(in_src), ptr(ws), ptr(err), st)
                return
            for src, dst in _edge_chunks(edge_index, chunk_edges, dev):
                L.grapes_graph_norm_add_edges(pass_, N, ptr(src), ptr(dst), int(src.numel()), ptr(self.in_off),
                                              ptr(in_src), ptr(ws), ptr(err), st)

        L.grapes_graph_norm_begin(N, ptr(ws), ws.numel(), ptr(err), st)
        run(0, None)
        L.grapes_graph_norm_offsets(N, ptr(ws), ptr(self.in_off), ptr(self.dinv), ptr(nnz), st)
        self._check(err)
        self.n, self.E = N, int(nnz.item())                      # one-off read-back: the size of in_src
        self.in_src = torch.empty(max(self.E, 1), dtype=torch.int32, device=dev)
        run(1, self.in_src)
        L.grapes_graph_norm_finish(N, ptr(self.in_off), ptr(self.in_src), ptr(ws), st)
        del ws
        if self.E == 0:
            self.in_src = self.in_src[:0]

    @staticmethod
    def _check(err, edges: str = "in-edges"):
        e = int(err.item())
        if e & 1:
            raise GrapesError("edge_index holds node ids outside [0, num_nodes)")
        if e & 2:
            raise GrapesError(f"a node has 2^31 - 1 or more {edges}")

    def aggregate_rows(self, x: torch.Tensor, slab: torch.Tensor, R: int, out: torch.Tensor, bias=None,
                       transpose: bool = False) -> torch.Tensor:
        """out[j] = (A_hat x)[r0 + j] (+ bias) for j < R, slab = int32 {R, r0} on the device; x fp32 or bf16 rows
        (widened on read), out fp32 [>= R, >= F] with a unit column stride.  ``transpose``: rows of A_hat^T x."""
        F = x.shape[1]
        if transpose:
            self.build_transposed()
        off, idx = (self.out_off, self.out_dst) if transpose else (self.in_off, self.in_src)
        lib().grapes_aggregate_rows64(self.holder.ctx, ptr(x), int(x.dtype == torch.bfloat16), F, x.stride(0), ptr(slab),
                                      R, ptr(off), ptr(idx), ptr(self.dinv), ptr(bias), ptr(out), out.stride(0),
                                      _stream())
        return out

    def aggregate(self, x: torch.Tensor, transpose: bool = False, bias=None) -> torch.Tensor:
        """A_hat x (+ bias) over all N rows, or A_hat^T x (+ bias) with ``transpose``: fp32 [N, F], one
        ``grapes_aggregate_rows64`` launch per slab of ``SLAB_ROWS`` rows (bit-identical to ``grapes_aggregate`` on the
        int32 structure of the same graph, see :class:`GraphNorm`)."""
        x = x.contiguous()
        out = torch.empty((self.n, x.shape[1]), dtype=torch.float32, device=x.device)
        if self._slabs is None:
            self._slabs = _slab_plan(0, self.n, self.SLAB_ROWS, x.device)
        for i, r0 in enumerate(self._slabs[0]):
            self.aggregate_rows(x, self._slabs[1][i], min(self.SLAB_ROWS, self.n - r0), out[r0:], bias, transpose)
        return out

    #: rows per launch of :meth:`aggregate`: 2^20 rows take the whole-graph launch shape of the row-slab kernels
    SLAB_ROWS = 1 << 20

    def build_transposed(self):
        """The transposed arrays ``out_off`` (int64) / ``out_dst``, once."""
        if self.out_off is None:
            edge_index, chunk_edges = self._input
            self.out_off, self.out_dst = transposed_structure(self.n, self.dinv.device, self.graph, edge_index,
                                                              chunk_edges)


def transposed_structure(N: int, dev, graph=None, edge_index=None, chunk_edges: int = 1 << 27):
    """(out_off int64 [N + 1], out_dst int32 [nnz']) of the transposed gcn_norm structure (``grapes_graph_norm_t_*``):
    row s lists the destinations of the edges s -> d, ascending, stored self-loops dropped, duplicates of ``edge_index``
    kept.  Read from ``edge_index`` (host or device int64 [2, E], in chunks of ``chunk_edges`` columns) when given,
    otherwise from ``graph``'s canonical CSR.  With the forward's ``dinv`` it is A_hat^T."""
    L, st = lib(), _stream()
    ws = torch.empty(max(int(L.cdll.grapes_graph_norm_workspace_bytes(N)), 1), dtype=torch.uint8, device=dev)
    err = torch.zeros(1, dtype=torch.int32, device=dev)
    nnz = torch.zeros(1, dtype=torch.int64, device=dev)
    out_off = torch.empty(N + 1, dtype=torch.int64, device=dev)

    def run(pass_, out_dst):
        if edge_index is None:
            L.grapes_graph_norm_t_add_csr(pass_, N, ptr(graph.indptr), ptr(graph.indices), 0, N, ptr(out_off),
                                          ptr(out_dst), ptr(ws), ptr(err), st)
            return
        for src, dst in _edge_chunks(edge_index, chunk_edges, dev):
            L.grapes_graph_norm_t_add_edges(pass_, N, ptr(src), ptr(dst), int(src.numel()), ptr(out_off), ptr(out_dst),
                                            ptr(ws), ptr(err), st)

    L.grapes_graph_norm_begin(N, ptr(ws), ws.numel(), ptr(err), st)
    run(0, None)
    L.grapes_graph_norm_t_offsets(N, ptr(ws), ptr(out_off), ptr(nnz), st)
    WideGraphNorm._check(err, "out-edges")
    E = int(nnz.item())                                          # one-off read-back: the size of out_dst
    out_dst = torch.empty(max(E, 1), dtype=torch.int32, device=dev)
    run(1, out_dst)
    if edge_index is not None:
        L.grapes_graph_norm_finish(N, ptr(out_off), ptr(out_dst), ptr(ws), st)
    del ws
    return out_off, (out_dst if E > 0 else out_dst[:0])


def _edge_chunks(edge_index, chunk_edges, dev):
    """(src, dst) int64 device slices of ``edge_index`` [2, E] (host or device), ``chunk_edges`` columns at a time."""
    for a in range(0, int(edge_index.shape[1]), chunk_edges):
        yield (edge_index[0, a:a + chunk_edges].to(device=dev, dtype=torch.int64).contiguous(),
               edge_index[1, a:a + chunk_edges].to(device=dev, dtype=torch.int64).contiguous())


class ShardedGraphNorm:
    """One rank's destination window of the :class:`WideGraphNorm` structure, for the data-parallel full-batch evaluation
    (:func:`full_graph_forward_sharded`).  The rows are cut into ``world`` contiguous windows ``bounds[r] .. bounds[r+1]``
    balanced by the prefix of indeg + 1 (``grapes_graph_norm_window_bounds``; every rank computes the same bounds, windows
    are empty when N < world).  Holds ``in_off`` int64 [rows + 1] local to the window, ``in_src`` int32 of the window's rows
    only (~1/world of the whole) and ``dinv`` fp32 for all N nodes (the source weights); equal bit for bit to rows
    ``lo .. hi`` of :class:`WideGraphNorm`.  Every degree is still counted (pass 0 reads the whole input); pass 1 scatters
    only the edges into the window.  Device memory beyond the outputs: the ~4 N-byte workspace, plus the full int64
    [N + 1] offsets until the window's are cut out, plus one chunk of a host edge list."""

    def __init__(self, graph, world: int, rank: int, edge_index=None, chunk_edges: int = 1 << 27):
        if not 0 <= rank < world:
            raise GrapesError(f"rank {rank} outside a world of {world}")
        dev = graph.device
        N = graph.num_nodes
        L, st = lib(), _stream()
        self.graph, self.world, self.rank = graph, int(world), int(rank)
        self.holder = _any_ctx(dev)
        self.n = N
        self._input = (edge_index, chunk_edges)
        self.out_off = self.out_dst = None
        ws = torch.empty(max(int(L.cdll.grapes_graph_norm_workspace_bytes(N)), 1), dtype=torch.uint8, device=dev)
        err = torch.zeros(1, dtype=torch.int32, device=dev)
        nnz = torch.zeros(1, dtype=torch.int64, device=dev)
        full = torch.empty(N + 1, dtype=torch.int64, device=dev)
        self.dinv = torch.empty(N, dtype=torch.float32, device=dev)
        L.grapes_graph_norm_begin(N, ptr(ws), ws.numel(), ptr(err), st)
        if edge_index is None:
            L.grapes_graph_norm_add_csr(0, N, ptr(graph.indptr), ptr(graph.indices), 0, N, None, None, ptr(ws), ptr(err), st)
        else:
            for src, dst in _edge_chunks(edge_index, chunk_edges, dev):
                L.grapes_graph_norm_add_edges(0, N, ptr(src), ptr(dst), int(src.numel()), None, None, ptr(ws), ptr(err), st)
        L.grapes_graph_norm_offsets(N, ptr(ws), ptr(full), ptr(self.dinv), ptr(nnz), st)
        bounds = torch.empty(self.world + 1, dtype=torch.int64, device=dev)
        L.grapes_graph_norm_window_bounds(N, ptr(full), self.world, ptr(bounds), st)
        WideGraphNorm._check(err)
        self.bounds = [int(b) for b in bounds.tolist()]                 # one-off read-back
        self.lo, self.hi = self.bounds[rank], self.bounds[rank + 1]
        self.rows = self.hi - self.lo
        self.in_off = (full[self.lo:self.hi + 1] - full[self.lo]).contiguous()
        del full
        self.E = int(self.in_off[-1].item())
        self.in_src = torch.empty(max(self.E, 1), dtype=torch.int32, device=dev)
        if edge_index is None:
            L.grapes_graph_norm_window_add_csr(N, ptr(graph.indptr), ptr(graph.indices), 0, N, self.lo, self.hi,
                                               ptr(self.in_off), ptr(self.in_src), ptr(ws), st)
        else:
            for src, dst in _edge_chunks(edge_index, chunk_edges, dev):
                L.grapes_graph_norm_window_add_edges(N, ptr(src), ptr(dst), int(src.numel()), self.lo, self.hi,
                                                     ptr(self.in_off), ptr(self.in_src), ptr(ws), st)
        if self.rows > 0:
            L.grapes_graph_norm_finish(self.rows, ptr(self.in_off), ptr(self.in_src), ptr(ws), st)
        del ws
        self._src = self.in_src                    # non-null for the kernels even when the window has no in-edge
        if self.E == 0:
            self.in_src = self.in_src[:0]

    def build_transposed(self):
        """The source window ``lo .. hi`` of the transposed structure, once, from the constructor's input: ``out_off``
        int64 [rows + 1] local to the window and ``out_dst`` int32 (``grapes_graph_norm_t_window_*``), equal bit for bit
        to rows ``lo .. hi`` of :func:`transposed_structure`.  The same bounds as the forward window, so a rank owns the
        same rows in both directions; ``dinv`` is not touched.  Device memory beyond the outputs: the ~4 N-byte workspace
        plus the full int64 [N + 1] offsets until the window's are cut out, plus one chunk of a host edge list."""
        if self.out_off is not None:
            return
        edge_index, chunk_edges = self._input
        graph, N, dev = self.graph, self.n, self.dinv.device
        L, st = lib(), _stream()
        ws = torch.empty(max(int(L.cdll.grapes_graph_norm_workspace_bytes(N)), 1), dtype=torch.uint8, device=dev)
        err = torch.zeros(1, dtype=torch.int32, device=dev)
        nnz = torch.zeros(1, dtype=torch.int64, device=dev)
        full = torch.empty(N + 1, dtype=torch.int64, device=dev)
        L.grapes_graph_norm_begin(N, ptr(ws), ws.numel(), ptr(err), st)
        if edge_index is None:
            L.grapes_graph_norm_t_add_csr(0, N, ptr(graph.indptr), ptr(graph.indices), 0, N, None, None, ptr(ws), ptr(err),
                                          st)
        else:
            for src, dst in _edge_chunks(edge_index, chunk_edges, dev):
                L.grapes_graph_norm_t_add_edges(0, N, ptr(src), ptr(dst), int(src.numel()), None, None, ptr(ws), ptr(err),
                                                st)
        L.grapes_graph_norm_t_offsets(N, ptr(ws), ptr(full), ptr(nnz), st)
        WideGraphNorm._check(err, "out-edges")
        out_off = (full[self.lo:self.hi + 1] - full[self.lo]).contiguous()
        del full
        E = int(out_off[-1].item())                                   # one-off read-back: the size of out_dst
        out_dst = torch.empty(max(E, 1), dtype=torch.int32, device=dev)
        if edge_index is None:
            L.grapes_graph_norm_t_window_add_csr(N, ptr(graph.indptr), ptr(graph.indices), 0, N, self.lo, self.hi,
                                                 ptr(out_off), ptr(out_dst), ptr(ws), st)
        else:
            for src, dst in _edge_chunks(edge_index, chunk_edges, dev):
                L.grapes_graph_norm_t_window_add_edges(N, ptr(src), ptr(dst), int(src.numel()), self.lo, self.hi,
                                                       ptr(out_off), ptr(out_dst), ptr(ws), st)
            if self.rows > 0:
                L.grapes_graph_norm_finish(self.rows, ptr(out_off), ptr(out_dst), ptr(ws), st)
        del ws
        self._dst = out_dst                        # non-null for the kernels even when the window has no out-edge
        self.out_off, self.out_dst = out_off, (out_dst if E > 0 else out_dst[:0])

    @property
    def in_off_base(self) -> int:
        """Device address that makes ``in_off[r]`` of the row-slab kernels (r = graph row) land on local row r - lo: the
        window's offsets shifted back by ``lo`` entries.  Only rows of the window are ever read through it."""
        return self.in_off.data_ptr() - 8 * self.lo

    def aggregate_rows(self, x: torch.Tensor, slab: torch.Tensor, R: int, out: torch.Tensor, bias=None) -> torch.Tensor:
        """:meth:`WideGraphNorm.aggregate_rows` for a slab {R, r0} inside the window (r0 a graph row): x holds ALL rows."""
        F = x.shape[1]
        lib().grapes_aggregate_rows64(self.holder.ctx, ptr(x), int(x.dtype == torch.bfloat16), F, x.stride(0), ptr(slab),
                                      R, self.in_off_base, ptr(self._src), ptr(self.dinv), ptr(bias), ptr(out),
                                      out.stride(0), _stream())
        return out

    def aggregate_rows_peer(self, z_table, slab: torch.Tensor, R: int, out: torch.Tensor, bias=None,
                            transpose: bool = False, F=None) -> torch.Tensor:
        """The same over Z partitioned by window: rank o's rows in ``z_table.ptrs[o]`` (pitch ``z_table.ld`` floats, the
        first ``F`` of them read, default all), ``grapes_aggregate_rows64_peer``; bit-identical to :meth:`aggregate_rows`
        over the unpartitioned Z.  ``transpose``: rows of A_hat^T Z on the transposed window (:meth:`build_transposed`,
        built here on first use), bit-identical to ``WideGraphNorm.aggregate(Z, transpose=True)``."""
        import ctypes
        F = z_table.ld if F is None else int(F)
        if transpose:
            self.build_transposed()
        off, idx = (self.out_off, self._dst) if transpose else (self.in_off, self._src)
        b = (ctypes.c_int64 * (self.world + 1))(*self.bounds)
        lib().grapes_aggregate_rows64_peer(self.holder.ctx, z_table.ptrs, b, self.world, F, z_table.ld, ptr(slab), R,
                                           off.data_ptr() - 8 * self.lo, ptr(idx), ptr(self.dinv), ptr(bias), ptr(out),
                                           out.stride(0), _stream())
        return out

    def aggregate_rows_sharded(self, ptrs, bounds_c, world: int, x_bf16: bool, F: int, ld: int, slab: torch.Tensor,
                               R: int, out: torch.Tensor, bias=None) -> torch.Tensor:
        """:meth:`aggregate_rows` over a table sharded by the feature bounds (``bounds_c``, HOST int64 [world + 1]):
        owner o's rows at ``ptrs[o]`` with pitch ``ld`` elements, fp32 or bf16 (``grapes_aggregate_rows64_peer_x``);
        bit-identical to :meth:`aggregate_rows` over the unpartitioned table."""
        lib().grapes_aggregate_rows64_peer_x(self.holder.ctx, ptrs, bounds_c, int(world), int(bool(x_bf16)), F, ld,
                                             ptr(slab), R, self.in_off_base, ptr(self._src), ptr(self.dinv), ptr(bias),
                                             ptr(out), out.stride(0), _stream())
        return out


def _gemm_into(A, lda, W, ldw, C, ldc, M, N, K, bias=None):
    """C[:M, :N] = A W^T (+ bias) on the same SIMT ``grapes_gemm`` call as :func:`_gemm` (layout 3), into a caller view."""
    if M > 0:
        lib().grapes_gemm(_any_ctx(A.device).ctx, 3, ptr(A), lda, ptr(W), ldw, ptr(C), ldc, None, M, N, K, ptr(bias), 0,
                          None, 0, _stream())


def slab_rows_for(n: int, per_row_bytes: int, resident_bytes: int, device, mem_budget=None, max_rows: int = 1 << 20) -> int:
    """Rows per slab that fit ``mem_budget`` bytes (default: free device memory, counting the blocks torch's allocator
    holds unused, less a margin of 5 % of the device and at least 2 GiB) after ``resident_bytes`` more are allocated, at
    most ``max_rows``: 2^20 rows already take the whole-graph launch shape of the aggregation (one CTA per SM, 32-entry
    chunks), and the slab temporaries stay ~1-2 GB."""
    if mem_budget is None:
        free, total = torch.cuda.mem_get_info(device)
        free += torch.cuda.memory_reserved(device) - torch.cuda.memory_allocated(device)
        mem_budget = free - max(total // 20, 2 << 30)
    rows = (int(mem_budget) - int(resident_bytes)) // max(int(per_row_bytes), 1)
    if rows < 1:
        raise GrapesError(f"streamed full-graph forward: {resident_bytes / 2**30:.1f} GiB resident leave no room for a slab "
                          f"within the memory budget of {mem_budget / 2**30:.1f} GiB")
    return int(min(rows, max_rows, max(n, 1)))


@torch.no_grad()
def full_graph_forward_streamed(gcn: "GCN", x: torch.Tensor, gn: WideGraphNorm, slab_rows=None, mem_budget=None,
                                y=None, mask=None, return_logits: bool = True):
    """``gcn_c(x, edge_index)`` over the whole graph (eval.py:50) for the two-layer classifier ``GCN(F, [D, C])``, one row
    slab at a time, on a :class:`WideGraphNorm`.  The products are those of ``gcn(x, GraphNorm)`` in the same order and on
    the same kernels, so the logits are bit-identical to it:

    * layer 1, F <= D: per slab Y = A_hat X (``aggregate_rows`` on the fp32 or bf16 rows as stored), H = relu(Y W1^T + b1);
      F > D: per slab P = X W1^T into a resident [N, D] array, then per slab H = relu(A_hat P + b1);
    * Z[slab] = H W2^T into ONE resident [N, round_up(C, 4)] array (zero pad columns); H never exists for all N;
    * per slab logits = A_hat Z + b2.

    ``slab_rows`` (default: what ``mem_budget`` allows, see :func:`slab_rows_for`) bounds the slab temporaries.  With ``y``
    (and ``mask``, default all rows) the scores of ``eval._scores`` are reduced per slab on the device.  Returns
    (logits [N, C] or None when ``return_logits`` is False, (accuracy, f1) or None).  Other depths, a layer 2 that would
    aggregate first (D <= C), other table dtypes and dropout in training mode raise ``GrapesError``."""
    w1, b1, w2, b2, D, C, C4 = _classifier_parts(gcn, x)
    dev = x.device
    N, F = x.shape                                    # (shadows torch.nn.functional inside this function)
    agg_first = F <= D
    resident = N * C4 * 4 + (0 if agg_first else N * D * 4) + (N * C4 * 4 if return_logits else 0)
    R = int(slab_rows) if slab_rows else slab_rows_for(N, _slab_row_bytes(x, D, C4), resident, dev, mem_budget)
    R = max(1, min(R, max(N, 1)))
    starts, slabs = _slab_plan(0, N, R, dev)
    Z = torch.zeros((N, C4), dtype=torch.float32, device=dev)
    _layer1_into(x, gn, (w1, b1, w2, D, C, C4), starts, slabs, N, R, Z, 0)
    logits, counts = _layer2(lambda s, n, o: gn.aggregate_rows(Z, s, n, o, bias=b2), starts, slabs, N, R, C, C4, dev,
                             y, mask, return_logits)
    scores = None if counts is None else _scores_from_counts(counts, y.dim() == 1)
    return logits, scores


def _is_sharded(x) -> bool:
    from .dist import ShardedFeatures
    return isinstance(x, ShardedFeatures)


def row_slab_refusal(gcn: "GCN", x):
    """Why the row-slab forwards (:func:`full_graph_forward_streamed`, :func:`full_graph_forward_sharded`) do not cover
    this classifier and feature table (a tensor or a :class:`grapes_b200.dist.ShardedFeatures`), or None when they do."""
    if _is_sharded(x):
        x = x.local
    layers = list(gcn.gcn_layers)
    if len(layers) != 2:
        return f"streamed full-graph forward covers the two-layer classifier, not {len(layers)} layers"
    if gcn.training and gcn.dropout > 0:
        return "streamed full-graph forward is evaluation only: dropout in training mode"
    if x.dtype not in (torch.float32, torch.bfloat16) or x.dim() != 2 or x.stride(1) != 1:
        return "streamed full-graph forward reads fp32 or bf16 rows with a unit column stride"
    if layers[0].lin.weight.shape[0] <= layers[1].lin.weight.shape[0]:
        return "streamed full-graph forward needs hidden width D > classes C (layer 2 transforms first)"
    return None


def _classifier_parts(gcn: "GCN", x: torch.Tensor):
    """Checks of the row-slab forwards and the classifier's fp32 weights: (w1, b1, w2, b2 padded to C4, D, C, C4)."""
    why = row_slab_refusal(gcn, x)
    if why is not None:
        raise GrapesError(why)
    layers = list(gcn.gcn_layers)
    w1 = layers[0].lin.weight.detach().float().contiguous()
    b1 = layers[0].bias.detach().float().contiguous()
    w2 = layers[1].lin.weight.detach().float().contiguous()
    D, C = w1.shape[0], w2.shape[0]
    C4 = (C + 3) // 4 * 4
    b2 = F_pad(layers[1].bias.detach().float(), C4 - C).contiguous()
    return w1, b1, w2, b2, D, C, C4


def _slab_row_bytes(x, D: int, C4: int) -> int:
    x = x.local if _is_sharded(x) else x
    F = x.shape[1]
    agg_first = F <= D
    return 4 * ((F if agg_first else 0) + (F if (not agg_first and x.dtype != torch.float32) else 0) + D + C4)


def _slab_plan(lo: int, hi: int, R: int, dev):
    """Slab starts over rows [lo, hi) and the device {rows, r0} pair of each."""
    starts = list(range(lo, hi, R))
    slabs = torch.tensor([[min(R, hi - r0), r0] for r0 in starts] or [[0, 0]], dtype=torch.int32, device=dev)
    return starts, slabs


def _layer1_into(x, gn, w, starts, slabs, hi, R, Z, z0, p_table=None):
    """Z[r - z0] = relu(A_hat X W1^T + b1)[r] W2^T for the rows r of the slabs (ending at ``hi``), at the narrower width:
    F <= D aggregates X per slab first; F > D forms P = X W1^T for ALL N rows (the sources of any row) first.  A sharded
    table ``x`` (:class:`grapes_b200.dist.ShardedFeatures`) is read from its owners; with F > D, P is then the sharded
    ``p_table`` (:func:`sharded_layer1_p`), already formed by every rank."""
    w1, b1, w2, D, C, C4 = w
    sharded = _is_sharded(x)
    dev = gn.dinv.device
    N, F = (x.N, x.F) if sharded else x.shape
    H = torch.empty((R, D), dtype=torch.float32, device=dev)
    if F <= D:
        Y = torch.empty((R, F), dtype=torch.float32, device=dev)
        for i, r0 in enumerate(starts):
            n = min(R, hi - r0)
            if sharded:
                gn.aggregate_rows_sharded(x.ptrs, x.bounds_c, x.world, x.x_bf16, F, x.ldx, slabs[i], n, Y)
            else:
                gn.aggregate_rows(x, slabs[i], n, Y)
            _gemm_into(Y, F, w1, F, H, D, n, D, F, bias=b1)
            torch.relu_(H[:n])
            _gemm_into(H, D, w2, D, Z[r0 - z0:], C4, n, C, D)
        del Y
    elif sharded:
        for i, r0 in enumerate(starts):
            n = min(R, hi - r0)
            gn.aggregate_rows_sharded(p_table.ptrs, x.bounds_c, x.world, False, D, p_table.ld, slabs[i], n, H, bias=b1)
            torch.relu_(H[:n])
            _gemm_into(H, D, w2, D, Z[r0 - z0:], C4, n, C, D)
    else:
        P = torch.empty((N, D), dtype=torch.float32, device=dev)
        for r0 in range(0, N, R):
            n = min(R, N - r0)
            xs = x[r0:r0 + n] if x.dtype == torch.float32 else x[r0:r0 + n].float()
            _gemm_into(xs, xs.stride(0), w1, F, P[r0:], D, n, D, F)
        for i, r0 in enumerate(starts):
            n = min(R, hi - r0)
            gn.aggregate_rows(P, slabs[i], n, H, bias=b1)
            torch.relu_(H[:n])
            _gemm_into(H, D, w2, D, Z[r0 - z0:], C4, n, C, D)
        del P
    del H


def _layer2(agg, starts, slabs, hi, R, C, C4, dev, y, mask, return_logits):
    """logits = A_hat Z + b2 per slab through ``agg(slab, n, out)``, with the masked counts of :func:`_slab_counts` reduced
    on the device when ``y`` is given.  Returns (logits [hi - starts[0], C] or None, counts int64 [3] or None)."""
    lo = starts[0] if starts else hi
    logits = torch.empty((hi - lo, C4), dtype=torch.float32, device=dev) if return_logits else None
    out = None if return_logits else torch.empty((R, C4), dtype=torch.float32, device=dev)
    counts = torch.zeros(3, dtype=torch.int64, device=dev) if y is not None else None
    for i, r0 in enumerate(starts):
        n = min(R, hi - r0)
        o = logits[r0 - lo:r0 - lo + n] if return_logits else out
        agg(slabs[i], n, o)
        if counts is not None:
            lg, ys = o[:n, :C], y[r0:r0 + n]
            if mask is not None:
                m = mask[r0:r0 + n]
                lg, ys = lg[m], ys[m]
            counts += _slab_counts(lg, ys)
    return (logits[:, :C] if return_logits else None), counts


class LocalRowTable:
    """A partitioned row table (the layer-2 operand of :func:`full_graph_forward_sharded`, or the shards of
    :class:`grapes_b200.dist.ShardedFeatures`) for one emulated rank of a single process: every
    window's rows in its own allocation on this device (``tables[o]``, shared by the emulated ranks), a barrier that does
    nothing.  Run :func:`sharded_layer1` for every emulated rank before :func:`sharded_layer2` for any of them.
    :class:`grapes_b200.dist.PeerRowTable` is the same interface over the ranks' symmetric memory."""

    def __init__(self, tables, rank: int):
        import ctypes
        self.tables, self.rank = tables, rank
        self.rows = tables[rank]
        self.ld = int(self.rows.shape[1])
        self.ptrs = (ctypes.c_void_p * len(tables))(*[t.data_ptr() for t in tables])

    @staticmethod
    def make(world: int, rows: int, ld: int, device, dtype: torch.dtype = torch.float32):
        tables = [torch.zeros((max(rows, 1), ld), dtype=dtype, device=device) for _ in range(world)]
        return [LocalRowTable(tables, r) for r in range(world)]

    def barrier(self):
        pass


def _sharded_rows(sgn, R):
    return max(1, min(int(R), max(sgn.rows, 1)))


def needs_p_table(gcn: "GCN", x) -> bool:
    """True when :func:`full_graph_forward_sharded` over the sharded table ``x`` needs a P table (F > D): a row table of
    ``x``'s bounds, [max rows, D] fp32 per rank, for :func:`sharded_layer1_p`."""
    return _is_sharded(x) and x.F > int(list(gcn.gcn_layers)[0].lin.weight.shape[0])


@torch.no_grad()
def sharded_layer1_p(gcn: "GCN", x, p_table, slab_rows=None, mem_budget=None):
    """Phase 0 of :func:`full_graph_forward_sharded` over a sharded feature table with F > D: P = X W1^T for this rank's
    table rows (``x.local``) into ``p_table.rows`` (pitch D), on the SIMT GEMM of the streamed forward, so P is
    bit-identical to its [N, D] P; layer 1 then aggregates P read from its owners.  Every rank's phase 0 must complete
    before any rank's phase 1."""
    w1, b1, w2, b2, D, C, C4 = _classifier_parts(gcn, x)
    rows, F = x.hi - x.lo, x.F
    if p_table.ld != D or p_table.rows.shape[0] < rows:
        raise GrapesError(f"P table of pitch {p_table.ld} x {p_table.rows.shape[0]} rows; the shard needs {D} x {rows}")
    dev = p_table.rows.device
    R = int(slab_rows) if slab_rows else slab_rows_for(rows, 4 * (F + D), 0, dev, mem_budget)
    R = max(1, min(R, max(rows, 1)))
    for a in range(0, rows, R):
        n = min(R, rows - a)
        xs = x.local[a:a + n] if x.dtype == torch.float32 else x.local[a:a + n].float()
        _gemm_into(xs, xs.stride(0), w1, F, p_table.rows[a:], D, n, D, F)


@torch.no_grad()
def sharded_layer1(gcn: "GCN", x, sgn: ShardedGraphNorm, z_table, slab_rows=None, mem_budget=None, p_table=None):
    """Phase 1 of :func:`full_graph_forward_sharded`: Z rows of this rank's window into ``z_table.rows`` (local row j =
    graph row lo + j), on the calls and in the order of :func:`full_graph_forward_streamed`'s layer 1.  ``x`` is the
    replicated table or a :class:`grapes_b200.dist.ShardedFeatures` (rows read from their owners,
    ``grapes_aggregate_rows64_peer_x``).  With F > D and a replicated table every rank forms P = X W1^T for ALL N rows
    (the sources of its window may be any rows), so that product and its [N, D] buffer do not shrink with the number of
    ranks; with a sharded table each rank forms P for its own table rows only (``p_table``, :func:`sharded_layer1_p`)."""
    w1, b1, w2, b2, D, C, C4 = _classifier_parts(gcn, x)
    if needs_p_table(gcn, x) and p_table is None:
        raise GrapesError("sharded feature table with F > D: layer 1 aggregates the sharded P = X W1^T (p_table)")
    if sgn.rows == 0:
        return
    if z_table.ld != C4 or z_table.rows.shape[0] < sgn.rows:
        raise GrapesError(f"row table of pitch {z_table.ld} x {z_table.rows.shape[0]} rows; the window needs {C4} x {sgn.rows}")
    sharded = _is_sharded(x)
    N, F = (x.N, x.F) if sharded else x.shape
    if sharded and (x.N != sgn.n or x.world != sgn.world):
        raise GrapesError(f"sharded table of {x.N} rows over {x.world} ranks; the structure has {sgn.n} over {sgn.world}")
    dev = sgn.dinv.device
    resident = 0 if (F <= D or sharded) else N * D * 4
    R = int(slab_rows) if slab_rows else slab_rows_for(sgn.rows, _slab_row_bytes(x, D, C4), resident, dev, mem_budget)
    R = _sharded_rows(sgn, R)
    starts, slabs = _slab_plan(sgn.lo, sgn.hi, R, dev)
    _layer1_into(x, sgn, (w1, b1, w2, D, C, C4), starts, slabs, sgn.hi, R, z_table.rows, sgn.lo, p_table)


@torch.no_grad()
def sharded_layer2(gcn: "GCN", sgn: ShardedGraphNorm, z_table, slab_rows=None, mem_budget=None, y=None, mask=None,
                   return_logits: bool = False):
    """Phase 2 of :func:`full_graph_forward_sharded`: logits of this rank's window = A_hat Z + b2 with Z read from the rows'
    owners (``ShardedGraphNorm.aggregate_rows_peer``).  Every rank's phase 1 must have completed.  Returns (window logits
    [rows, C] or None, int64 counts [3] of :func:`_slab_counts` or None)."""
    layers = list(gcn.gcn_layers)
    C = layers[1].lin.weight.shape[0]
    C4 = (C + 3) // 4 * 4
    b2 = F_pad(layers[1].bias.detach().float(), C4 - C).contiguous()
    dev = sgn.dinv.device
    resident = sgn.rows * C4 * 4 if return_logits else 0
    R = int(slab_rows) if slab_rows else slab_rows_for(sgn.rows, 4 * C4, resident, dev, mem_budget)
    R = _sharded_rows(sgn, R)
    starts, slabs = _slab_plan(sgn.lo, sgn.hi, R, dev)
    return _layer2(lambda s, n, o: sgn.aggregate_rows_peer(z_table, s, n, o, bias=b2), starts, slabs, sgn.hi, R, C, C4,
                   dev, y, mask, return_logits)


@torch.no_grad()
def full_graph_forward_sharded(gcn: "GCN", x, sgn: ShardedGraphNorm, z_table, y=None, mask=None,
                               return_logits: bool = False, slab_rows=None, mem_budget=None, p_table=None):
    """The data-parallel form of :func:`full_graph_forward_streamed`: this rank computes the rows of its window only.
    Layer 1 over the window's slabs (X replicated) writes Z for the window into this rank's slot of ``z_table``
    (``rows``, ``ld`` = round_up(C, 4), ``ptrs`` = every rank's slot, ``barrier()``); after a barrier, layer 2 aggregates the
    window reading each source row of Z from the rank that owns it; a second barrier keeps Z until every rank has read it.
    The window's logits are bit-identical to the same rows of :func:`full_graph_forward_streamed` and of ``gcn(x,
    GraphNorm)``.  Returns (window logits [rows, C] or None, int64 counts [3] of the window's masked rows or None); sum the
    counts over the ranks and score them with :func:`_scores_from_counts`.  ``x`` may be a sharded feature table
    (:class:`grapes_b200.dist.ShardedFeatures`, the same bounds on every rank); with F > D it needs ``p_table``
    (:func:`needs_p_table`), formed first by :func:`sharded_layer1_p` and followed by a barrier."""
    if needs_p_table(gcn, x):
        sharded_layer1_p(gcn, x, p_table, slab_rows=slab_rows, mem_budget=mem_budget)
        p_table.barrier()
    sharded_layer1(gcn, x, sgn, z_table, slab_rows=slab_rows, mem_budget=mem_budget, p_table=p_table)
    z_table.barrier()
    res = sharded_layer2(gcn, sgn, z_table, slab_rows=slab_rows, mem_budget=mem_budget, y=y, mask=mask,
                         return_logits=return_logits)
    z_table.barrier()
    return res


def _slab_counts(logits_masked: torch.Tensor, y_masked: torch.Tensor) -> torch.Tensor:
    """(argmax hits, rows, 0) single-label or (tp, fp, fn) multi-label of one slab's masked rows, on the device."""
    if y_masked.dim() == 1:
        hits = (torch.argmax(logits_masked, dim=1) == y_masked).sum()
        return torch.stack([hits, hits.new_tensor(y_masked.shape[0]), hits.new_zeros(())])
    y_pred = logits_masked > 0
    y_true = y_masked > 0.5
    return torch.stack([(y_true & y_pred).sum(), (~y_true & y_pred).sum(), (y_true & ~y_pred).sum()])


def _scores_from_counts(counts: torch.Tensor, single_label: bool):
    """(accuracy, f1) from the summed slab counts, with the arithmetic of ``eval._scores``."""
    a, b, c = (int(v) for v in counts.tolist())
    if single_label:
        acc = (torch.tensor(a, dtype=torch.float32) / b).item()      # float32 mean of the hit vector
        return acc, acc
    tp, fp, fn = a, b, c
    try:
        precision, recall = tp / (tp + fp), tp / (tp + fn)
        f1 = 2 * (precision * recall) / (precision + recall)
    except ZeroDivisionError:
        f1 = 0.
    return f1, f1


def dense_bias_relu_tc(Y: torch.Tensor, weight: torch.Tensor, bias: torch.Tensor) -> torch.Tensor:
    """relu(Y W^T + b) for a tall Y [n, K] on the tcgen05 kernels (3xTF32, fp32-accurate; ``grapes_gemm_bias_relu_tc``): the
    hidden layer of the whole-graph evaluation forward.  Requires out_features % 128 == 0 (<= 512)."""
    holder = _any_ctx(Y.device)
    L, ctx, st = lib(), holder.ctx, _stream()
    n, K = Y.shape
    D = weight.shape[0]
    ldy = Y.stride(0)
    assert Y.stride(1) == 1 and ldy % 4 == 0 and Y.data_ptr() % 16 == 0
    ldw = (K + 3) // 4 * 4
    w = weight.detach().float().contiguous()
    Wh = torch.empty((D, ldw), dtype=torch.float32, device=Y.device)
    Wl = torch.empty((D, ldw), dtype=torch.float32, device=Y.device)
    L.grapes_split_tf32(ctx, ptr(w), K, D, K, ptr(Wh), ptr(Wl), ldw, st)
    H = torch.empty((n, D), dtype=torch.float32, device=Y.device)
    cnt = torch.tensor([n], dtype=torch.int32, device=Y.device)
    b = bias.detach().float().contiguous()
    L.grapes_gemm_bias_relu_tc(ctx, ptr(Y), ldy, cnt.data_ptr(), n, K, ptr(Wh), ptr(Wl), ldw, D, ptr(b), ptr(H), D, st)
    return H


@torch.no_grad()
def full_graph_forward(gcn: "GCN", x: torch.Tensor, gn: GraphNorm) -> torch.Tensor:
    """``gcn_c(x, edge_index)`` over the whole graph (eval.py:50) for the two-layer classifier, forward only, every product on
    this library's kernels: Y = A_hat X (TMA-staged SpMM at the narrower width), H = relu(Y W1^T + b1) on the tensor cores,
    Z = H W2^T, logits = A_hat Z + b2.  Falls back to the module's own forward for other depths / hidden widths."""
    layers = list(gcn.gcn_layers)
    D = layers[0].lin.weight.shape[0] if layers else 0
    if len(layers) != 2 or D % 128 != 0 or D > 512 or x.shape[0] < 4096 or gcn.training and gcn.dropout > 0:
        return gcn(x, gn)[0]
    n, F = x.shape
    xp = x.float()
    if F % 4 != 0:                                    # 16-byte rows for the TMA-staged aggregation and the A tiles
        xp = torch.zeros((n, (F + 3) // 4 * 4), dtype=torch.float32, device=x.device)
        xp[:, :F].copy_(x)
        Y = gn.aggregate(xp)
    else:
        Y = gn.aggregate(xp.contiguous())
    H = dense_bias_relu_tc(Y[:, :F] if Y.shape[1] != F else Y, layers[0].lin.weight, layers[0].bias)
    w2 = layers[1].lin.weight.detach().float().contiguous()
    C = w2.shape[0]
    C4 = (C + 3) // 4 * 4
    Z = _gemm(3, H, D, w2, D, n, C, D, ldc=C4) if C4 != C else _gemm(3, H, D, w2, D, n, C, D)
    b2 = layers[1].bias.detach().float()
    if C4 != C:
        b2 = F_pad(b2, C4 - C)
    return gn.aggregate(Z, bias=b2.contiguous())[:, :C]


def F_pad(t: torch.Tensor, k: int) -> torch.Tensor:
    return F.pad(t, (0, k))


def _gemm(layout, A, lda, B, ldb, M, N, K, bias=None, relu=0, ldc=None):
    holder = _any_ctx(A.device)
    ldc = N if ldc is None else ldc
    C = torch.empty((M, N), dtype=torch.float32, device=A.device) if ldc == N else \
        torch.zeros((M, ldc), dtype=torch.float32, device=A.device)
    if M > 0:
        lib().grapes_gemm(holder.ctx, layout, ptr(A), lda, ptr(B), ldb, ptr(C), ldc, None, M, N, K, ptr(bias), relu,
                          None, 0, _stream())
    return C


def _gemm_tn(A, B, R, M, N):
    holder = _any_ctx(A.device)
    out = torch.zeros((M, N), dtype=torch.float32, device=A.device)
    if R > 0:
        lib().grapes_gemm_tn(holder.ctx, ptr(A), M, ptr(B), N, None, R, M, N, 1.0, 0, ptr(out), _stream())
    return out


def _colsum(M):
    """sum over the rows of M [R, C] (fp32, contiguous): ``grapes_colsum``, fixed-order slabs."""
    R, C = M.shape
    out = torch.zeros(C, dtype=torch.float32, device=M.device)
    if R > 0:
        n = torch.tensor([R], dtype=torch.int32, device=M.device)
        lib().grapes_colsum(_any_ctx(M.device).ctx, ptr(M), n.data_ptr(), R, C, C, 1.0, 0, ptr(out), _stream())
    return out


def gcn_structure(edge_index, num_nodes: int, device):
    """The gcn_norm structure GCNConv aggregates over for a raw ``edge_index`` [2, E] on ``num_nodes`` nodes (PyG
    semantics: duplicates counted, stored self-loops replaced by one per node).  Edge lists within the library's small
    context take :class:`NormAdj`; larger ones (the whole graph) :class:`WideGraphNorm`, built from the edge list in
    chunks (host or device).  Structures (:class:`NormAdj`, :class:`GraphNorm`, :class:`WideGraphNorm`) pass through."""
    if isinstance(edge_index, (NormAdj, WideGraphNorm)):
        return edge_index
    if max(int(edge_index.shape[1]), int(num_nodes), 1) > _any_ctx(device).max_frontier:
        return WideGraphNorm(None, edge_index=edge_index, num_nodes=num_nodes, device=device)
    return NormAdj(edge_index, num_nodes)


class _GCNConvFn(torch.autograd.Function):
    """out = A_hat (x W^T) + b, computed at the narrower width: (A_hat x) W^T when in <= out."""

    @staticmethod
    def forward(ctx_, x, weight, bias, adj: NormAdj):
        x = x.contiguous().float()
        w = weight.contiguous().float()
        n, I = x.shape
        O = w.shape[0]
        ctx_.adj, ctx_.agg_first = adj, I <= O
        if ctx_.agg_first:
            y = adj.aggregate(x)
            out = _gemm(3, y, I, w, I, n, O, I, bias=bias)
            ctx_.save_for_backward(y, w)
        else:
            O4 = (O + 3) // 4 * 4
            if O4 != O and n >= 4096:                                 # float4 / TMA aggregation path: pad the width
                h = _gemm(3, x, I, w, I, n, O, I, ldc=O4)
                b4 = None if bias is None else F.pad(bias.detach().float(), (0, O4 - O))
                out = adj.aggregate(h, bias=b4)[:, :O]
            else:
                h = _gemm(3, x, I, w, I, n, O, I)
                out = adj.aggregate(h, bias=bias)
            ctx_.save_for_backward(x, w)
        return out

    @staticmethod
    def backward(ctx_, dout):
        saved, w = ctx_.saved_tensors
        adj = ctx_.adj
        dout = dout.contiguous().float()
        n, O = dout.shape
        I = w.shape[1]
        need_dx = ctx_.needs_input_grad[0]
        db = _colsum(dout) if ctx_.needs_input_grad[2] else None
        dx = None
        if ctx_.agg_first:
            dW = _gemm_tn(dout, saved, n, O, I)                       # dout^T (A_hat x)
            if need_dx:
                dy = _gemm(1, dout, O, w, I, n, I, O)                # dout W
                dx = adj.aggregate(dy, transpose=True)
        else:
            dh = adj.aggregate(dout, transpose=True)                  # A_hat^T dout
            dW = _gemm_tn(dh, saved, n, O, I)
            if need_dx:
                dx = _gemm(1, dh, O, w, I, n, I, O)
        return dx, dW, db, None


class _Lin(nn.Module):
    def __init__(self, in_channels: int, out_channels: int):
        super().__init__()
        self.weight = nn.Parameter(torch.empty(out_channels, in_channels))


class GCNConv(nn.Module):
    """PyG 2.5.2 ``GCNConv(in, out)`` with default arguments (improved=False, cached=False,
    add_self_loops=True, normalize=True, bias=True); glorot weight, zero bias."""

    def __init__(self, in_channels: int, out_channels: int):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.lin = _Lin(in_channels, out_channels)
        self.bias = nn.Parameter(torch.zeros(out_channels))
        self.reset_parameters()

    def reset_parameters(self):
        a = math.sqrt(6.0 / (self.in_channels + self.out_channels))
        with torch.no_grad():
            self.lin.weight.uniform_(-a, a)
            self.bias.zero_()

    def forward(self, x, edge_index):
        """``edge_index``: a raw [2, E] edge list (see :func:`gcn_structure`) or a prebuilt structure; forward and
        backward (weights, bias and ``x`` when it requires grad) run on the library's kernels either way."""
        return _GCNConvFn.apply(x, self.lin.weight, self.bias, gcn_structure(edge_index, x.shape[0], x.device))


class GCN(nn.Module):
    def __init__(self, in_features: int, hidden_dims: List[int], dropout: float = 0.):
        super(GCN, self).__init__()
        self.dropout = dropout
        dims = [in_features] + hidden_dims
        gcn_layers = []
        for i in range(len(hidden_dims) - 1):
            gcn_layers.append(GCNConv(in_channels=dims[i], out_channels=dims[i + 1]))
        gcn_layers.append(GCNConv(in_channels=dims[-2], out_channels=dims[-1]))
        self.gcn_layers = nn.ModuleList(gcn_layers)

    def forward(self, x: torch.Tensor, edge_index: Union[torch.Tensor, List[torch.Tensor]]):
        layerwise_adjacency = type(edge_index) == list
        if not layerwise_adjacency:
            edge_index = gcn_structure(edge_index, x.shape[0], x.device)      # built once, shared by the layers
        for i, layer in enumerate(self.gcn_layers[:-1], start=1):
            edges = edge_index[-i] if layerwise_adjacency else edge_index
            x = torch.relu(layer(x, edges))
            x = F.dropout(x, p=self.dropout, training=self.training)
        edges = edge_index[0] if layerwise_adjacency else edge_index
        logits = self.gcn_layers[-1](x, edges)
        logits = F.dropout(logits, p=self.dropout, training=self.training)
        memory_alloc = torch.cuda.memory_allocated() / (1024 * 1024)
        return logits, memory_alloc
