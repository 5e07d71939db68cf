"""Drop-in mirror of the reference's ``eval.py`` (/root/reference/eval.py:11-165): same ``evaluate`` signature,
same two modes, same return ``(accuracy, f1)``.

* ``full_batch=True`` (the default of every reference config, eval.py:47-70): ONE forward of the classifier over the
  whole graph.  The reference moves the model to the CPU for this (``eval_on_cpu=True``, main.py:43); here it stays
  on the B200 -- the whole-graph aggregation is ``grapes_aggregate`` (TMA-staged SpMM, csrc/spmm_tma.cu) on the
  gcn_norm structure of the full CSR (:class:`grapes_b200.gcn.GraphNorm`, built once and cached on the graph).  From
  ``WIDE_MIN_EDGES`` edges on, the structure has int64 offsets (:class:`grapes_b200.gcn.WideGraphNorm`) and the forward
  runs over row slabs (:func:`grapes_b200.gcn.full_graph_forward_streamed`): same logits, bounded memory.
* ``full_batch=False`` (eval.py:71-163): every batch runs on the training engine's kernels, forward only
  (``GrapesEngine.predict``): frontier expansion, bitmap dedup / relabel, fused gather + aggregation, the sampler GCN's
  tcgen05 forward, DETERMINISTIC top-k on the probabilities (eval.py:126-130, ``GRAPES_NOISE_NONE_TOPK_PROBS``), the
  evaluation's block direction ``slice_adjacency(rows=previous_nodes, cols=batch_nodes)`` (eval.py:140-142, a filter of
  the hop's own row expansion), classifier forward, argmax of the target rows.  Batches are enqueued back to back
  (CUDA-graph replays); the host synchronises once, after the last batch.

``eval_on_cpu`` is accepted for signature compatibility and ignored: there is no CPU fallback (north_star).
sklearn's accuracy / micro-F1 on single-label predictions are both the fraction of correct predictions, computed
on the device.
"""
from __future__ import annotations

import os
from typing import Optional, Tuple

import warnings

import numpy as np
import torch
import torch.distributed as dist

from ._lib import GrapesError
from .gcn import (GCN, GraphNorm, ShardedGraphNorm, WideGraphNorm, _scores_from_counts, full_graph_forward,
                  full_graph_forward_sharded, full_graph_forward_streamed, needs_p_table, row_slab_refusal)
from .graph import DeviceGraph
from .utils import TensorMap, get_logger

# Edge count from which the full-batch evaluation runs on the int64 structure (WideGraphNorm) and the row-slab forward
# (full_graph_forward_streamed): the int32 offsets of GraphNorm and grapes_aggregate hold fewer entries.
WIDE_MIN_EDGES = (1 << 31) - 1


def _graph_norm(adjacency: DeviceGraph, data, wide: bool = False):
    """gcn_norm structure of ``data.edge_index`` (what eval.py:50 feeds GCNConv), cached on the graph object."""
    ei = getattr(data, "edge_index", None)
    key = (None if ei is None else (ei.data_ptr(), tuple(ei.shape)), wide)
    cached = getattr(adjacency, "_graph_norm", None)
    if cached is None or cached[0] != key:
        adjacency._graph_norm = None                                  # the previous structure goes before the new one is built
        cached = (key, (WideGraphNorm if wide else GraphNorm)(adjacency, edge_index=ei))
        adjacency._graph_norm = cached
    return cached[1]


def _scores(logits_masked: torch.Tensor, y_masked: torch.Tensor) -> Tuple[float, float]:
    if y_masked.dim() == 1:                                           # eval.py:51-55
        acc = (torch.argmax(logits_masked, dim=1) == y_masked).float().mean().item()
        return acc, acc                                               # micro-F1 == accuracy (single label)
    y_pred = logits_masked > 0                                        # eval.py:57-70
    y_true = y_masked > 0.5
    tp = int((y_true & y_pred).sum()); fp = int((~y_true & y_pred).sum()); fn = int((y_true & ~y_pred).sum())
    try:
        precision, recall = tp / (tp + fp), tp / (tp + fn)
        f1 = 2 * (precision * recall) / (precision + recall)
    except ZeroDivisionError:
        f1 = 0.
    return f1, f1


@torch.inference_mode()
def evaluate(gcn_c: GCN,
             gcn_gf: Optional[GCN],
             data,
             args,
             adjacency: DeviceGraph,
             node_map: Optional[TensorMap],
             num_indicators: int,
             device: torch.device,
             mask: torch.Tensor = None,
             eval_on_cpu: bool = True,
             loader=None,
             full_batch: bool = False,
             return_predictions: bool = False,
             engine=None,
             group=None,
             *,
             features=None,
             ):
    """``group``: a ``torch.distributed`` process group of more than one rank makes the evaluation data parallel, with
    the scores of one process (see :func:`_evaluate_sharded`); None or a one-rank group runs the single-process code.

    ``features``: the feature table sharded across the ranks of ``group`` (:class:`grapes_b200.dist.ShardedFeatures`),
    read instead of ``data.x``, which is then never moved to the device.  Mini batch runs on the engine (built over the
    sharded table when ``engine`` is None).  Full batch needs ``group`` and runs the sharded forward only: a classifier the
    row-slab forward does not cover, or a Z / P table that could not be mapped, raises ``GrapesError`` on every rank,
    since there is no replicated table to fall back to."""
    get_logger().info('Evaluating')
    device = torch.device(device)
    sharded_group = group is not None and dist.is_initialized() and dist.get_world_size(group) > 1
    if features is not None and full_batch and not sharded_group:
        raise GrapesError("full-batch evaluation of a sharded feature table runs over the process group that holds the "
                          "shards (pass group=); evaluate mini-batch (full_batch=False) otherwise")
    if device.type != "cuda":
        raise GrapesError("grapes_b200 has no CPU fallback: evaluation runs on the CUDA device (eval_on_cpu is ignored)")
    x = features if features is not None else data.x.to(device)
    y = data.y.to(device)
    gcn_c = gcn_c.to(device).eval()
    mask_d = mask.to(device) if mask is not None else torch.ones(data.num_nodes, dtype=torch.bool, device=device)
    if sharded_group:
        res = _evaluate_sharded(gcn_c, gcn_gf, data, args, adjacency, num_indicators, device, x, y, mask_d, loader,
                                full_batch, return_predictions, engine, group)
        if res is not None:
            return res

    if full_batch:
        ei = getattr(data, "edge_index", None)
        if (int(ei.shape[1]) if ei is not None else adjacency.nnz) >= WIDE_MIN_EDGES:
            # past 2^31 edges: int64 structure, row slabs, masked scores reduced per slab; [N, C] logits only on request
            logits_total, res = full_graph_forward_streamed(gcn_c, x, _graph_norm(adjacency, data, wide=True), y=y,
                                                            mask=mask_d, return_logits=return_predictions)
            return (res + (logits_total,)) if return_predictions else res
        # eval.py:50.  GRAPES_EVAL_TC=1: the fused whole-graph forward with its hidden layer on the tensor cores
        # (gcn.full_graph_forward; written after this round's GPU budget was spent, measured by bench.py's full_graph_eval leg)
        if os.environ.get("GRAPES_EVAL_TC", "0") == "1":
            logits_total = full_graph_forward(gcn_c, x, _graph_norm(adjacency, data))
        else:
            logits_total, _ = gcn_c(x, _graph_norm(adjacency, data))
        res = _scores(logits_total[mask_d], y[mask_d])
        return (res + (logits_total,)) if return_predictions else res

    # ---- mini-batch message passing (eval.py:71-163) on the engine's device path ----
    assert loader is not None, 'loader must be provided if full_batch is False'
    batches = [b[0] if isinstance(b, (tuple, list)) else b for b in loader]
    eng = engine if engine is not None else _eval_engine(adjacency, data, args, gcn_c, gcn_gf, num_indicators, device,
                                                         max([int(b.numel()) for b in batches] + [1]), x)
    total = sum(int(b.numel()) for b in batches)
    preds = torch.zeros(max(total, 1), dtype=torch.int32, device=device)
    off = 0
    for b in batches:                                                  # every batch is enqueued; nothing is read back
        n = int(b.numel())
        eng.predict(b.to(device), preds[off:off + n])
        off += n
    eng.check_overflow()                                               # the one synchronisation of the evaluation
    all_predictions = preds[:total].to(torch.int64)
    targets = y[mask_d]
    acc = (all_predictions == targets).float().mean().item()          # accuracy_score == micro f1_score here
    return (acc, acc, all_predictions) if return_predictions else (acc, acc)


def _mean_of_hits(hits: int, rows: int) -> float:
    """``(pred == y).float().mean().item()`` on the device from the integer count: CUDA's mean is the float32 sum times
    float32(1 / rows).  The float32 sum of a 0/1 vector is exact below 2^24 rows, so below that the result is bit for bit
    the one-process score; past it the one-process sum may round and the two can differ in the last place (the integer
    count here is the exact one)."""
    with np.errstate(divide="ignore", invalid="ignore"):
        return float(np.float32(hits) * (np.float32(1) / np.float32(rows)))


def _sharded_eval(adjacency: DeviceGraph, data, group, C4: int, device, p_shape=None, fallback: bool = True):
    """(window structure, peer row table or None, P table or None) of this rank, cached on the graph object like
    ``_graph_norm``.  The tables are None when the symmetric mapping failed on any rank (every rank agrees, so none of
    them waits on a peer).  ``p_shape`` = (rows, D): also the P table of a sharded feature table with F > D.
    ``fallback``: the caller runs the replicated evaluation when they are None (warned here)."""
    from .dist import PeerRowTable, ranks_agree
    ei = getattr(data, "edge_index", None)
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    key = (None if ei is None else (ei.data_ptr(), tuple(ei.shape)), world, rank, C4, p_shape)
    cached = getattr(adjacency, "_sharded_eval", None)
    if cached is None or cached[0] != key:
        adjacency._sharded_eval, adjacency._sharded_eval_p = None, None
        sgn, table, ptab, why = None, None, None, ""
        try:                                           # rank-local failures (memory, ids, mapping) become the fall-back
            sgn = ShardedGraphNorm(adjacency, world, rank, edge_index=ei)
            rows = max(sgn.bounds[r + 1] - sgn.bounds[r] for r in range(world))
            table = PeerRowTable(rows, C4, device, group)
            if p_shape is not None:
                ptab = PeerRowTable(p_shape[0], p_shape[1], device, group)
        except Exception as exc:                       # noqa: BLE001 -- reported below, never silent
            why, table = f"{type(exc).__name__}: {exc}", None
        if ranks_agree(table is not None, device, group):
            try:
                table.rendezvous()
                if ptab is not None:
                    ptab.rendezvous()
            except Exception as exc:                   # noqa: BLE001
                why, table = f"{type(exc).__name__}: {exc}", None
            if not ranks_agree(table is not None, device, group):
                table = None
        else:
            table = None
        if table is None:
            sgn, ptab = None, None                     # the replicated evaluation builds the whole structure instead
            adjacency._sharded_eval_failure = why or "on another rank"
            if fallback:
                warnings.warn("grapes_b200: sharded full-batch structure or peer-mapped row table unavailable" +
                              (f" ({why})" if why else
                              " on another rank") + "; every rank runs the replicated full-batch evaluation")
        cached = (key, sgn, table)
        adjacency._sharded_eval, adjacency._sharded_eval_p = cached, ptab
    return cached[1], cached[2], adjacency._sharded_eval_p


def _evaluate_sharded(gcn_c, gcn_gf, data, args, adjacency, num_indicators, device, x, y, mask_d, loader, full_batch,
                      return_predictions, engine, group):
    """Data-parallel evaluation over the ranks of ``group``, with the scores one process computes:

    * full batch: every rank builds its destination window of the structure (:class:`ShardedGraphNorm`) and runs
      :func:`full_graph_forward_sharded` (layer 2 reads Z over peer memory); the integer counts are summed over the ranks.
      ``return_predictions`` raises ``GrapesError`` (gathering [N, C] on every rank is the memory this path saves), and
      ``GRAPES_EVAL_TC`` has no effect.  Returns None -- the caller then runs the replicated evaluation -- when the
      row-slab forward does not cover the classifier (:func:`grapes_b200.gcn.row_slab_refusal`; weights and features are
      replicated, so every rank decides alike) or when the window structure or the peer mapping failed on any rank.
    * mini batch: rank r runs the batches i = r mod W of the split, all of them; hits and rows are summed as integers, and
      ``return_predictions`` gathers every rank's predictions back into batch order."""
    from .dist import ShardedFeatures, allreduce_counts_, eval_batches, gather_batch_predictions, ranks_agree
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    sharded_x = isinstance(x, ShardedFeatures)
    if full_batch:
        if return_predictions:
            raise GrapesError("data-parallel full-batch evaluation returns scores only: gathering the [N, C] logits on "
                              "every rank is the memory it avoids (evaluate without a group for the logits)")
        why = row_slab_refusal(gcn_c, x)
        if why is not None:
            if sharded_x:             # no replicated table to fall back to; the same decision on every rank
                raise GrapesError(f"full-batch evaluation of a sharded feature table: {why}; evaluate mini-batch "
                                  "(full_batch=False) instead")
            return None               # a classifier the row-slab forward does not cover: the same on every rank
        if sharded_x and (x.world != world or x.N != adjacency.num_nodes):
            raise GrapesError(f"sharded feature table of {x.N} rows over {x.world} ranks; the group has {world} ranks "
                              f"and the graph {adjacency.num_nodes} nodes")
        C = int(gcn_c.gcn_layers[-1].lin.weight.shape[0])
        p_shape = None
        if needs_p_table(gcn_c, x):
            p_shape = (max(x.bounds[r + 1] - x.bounds[r] for r in range(world)),
                       int(gcn_c.gcn_layers[0].lin.weight.shape[0]))
        sgn, table, ptab = _sharded_eval(adjacency, data, group, (C + 3) // 4 * 4, device, p_shape,
                                         fallback=not sharded_x)
        if table is None:
            if sharded_x:
                raise GrapesError("full-batch evaluation of a sharded feature table: window structure or peer-mapped "
                                  f"Z / P table unavailable ({adjacency._sharded_eval_failure}); evaluate mini-batch "
                                  "(full_batch=False) instead")
            return None
        _, counts = full_graph_forward_sharded(gcn_c, x, sgn, table, y=y, mask=mask_d, p_table=ptab)
        allreduce_counts_(counts, group)
        ei = getattr(data, "edge_index", None)
        if y.dim() == 1 and (int(ei.shape[1]) if ei is not None else adjacency.nnz) < WIDE_MIN_EDGES:
            acc = _mean_of_hits(int(counts[0]), int(counts[1]))       # what _scores computes on one GPU
            return acc, acc
        return _scores_from_counts(counts, y.dim() == 1)

    assert loader is not None, 'loader must be provided if full_batch is False'
    batches = [b[0] if isinstance(b, (tuple, list)) else b for b in loader]
    sizes = [int(b.numel()) for b in batches]
    mine = eval_batches(len(batches), rank, world)
    eng = engine if engine is not None else _eval_engine(adjacency, data, args, gcn_c, gcn_gf, num_indicators, device,
                                                         max(sizes + [1]), x)
    total = sum(sizes[i] for i in mine)
    preds = torch.zeros(max(total, 1), dtype=torch.int32, device=device)
    off = 0
    for i in mine:
        eng.predict(batches[i].to(device), preds[off:off + sizes[i]])
        off += sizes[i]
    failure = None
    try:
        eng.check_overflow()
    except GrapesError as exc:                         # raised on every rank, so none of them waits in the all-reduce
        failure = exc
    if not ranks_agree(failure is None, device, group):
        raise failure or GrapesError("data-parallel mini-batch evaluation: another rank's batches overflowed")
    local = preds[:total].to(torch.int64)
    targets = y[torch.cat([batches[i].to(device).long() for i in mine])] if mine else local
    counts = torch.stack([(local == targets).sum(), local.new_tensor(total)])
    allreduce_counts_(counts, group)
    acc = _mean_of_hits(int(counts[0]), int(counts[1]))
    if return_predictions:
        return acc, acc, gather_batch_predictions(local, sizes, group)
    return acc, acc


def _eval_engine(adjacency: DeviceGraph, data, args, gcn_c: GCN, gcn_gf: GCN, num_indicators: int, device, batch_size: int,
                 x=None):
    """Engine for a stand-alone ``evaluate(..., full_batch=False)`` call (the training loop passes its own): built once
    per (graph, features, shape) and cached on the graph object; the modules' weights are loaded on every call.  ``x``: the
    device table or a sharded one (default ``data.x``)."""
    from .dist import ShardedFeatures
    from .engine import GrapesEngine
    D = int(gcn_c.gcn_layers[0].lin.weight.shape[0])
    C = int(gcn_c.gcn_layers[-1].lin.weight.shape[0])
    if not isinstance(x, ShardedFeatures):
        x = data.x.to(device).contiguous()
        xkey = (x.data_ptr(), tuple(x.shape))
    else:
        xkey = (id(x), x.N, x.F)
    key = (xkey, D, C, int(batch_size), int(args.num_samples), int(args.sampling_hops), bool(num_indicators))
    cached = getattr(adjacency, "_eval_engine", None)
    if cached is None or cached[0] != key:
        eng = GrapesEngine(adjacency, x, data.y.to(device), num_classes=C, batch_size=int(batch_size),
                           num_samples=int(args.num_samples), sampling_hops=int(args.sampling_hops),
                           use_indicators=bool(num_indicators), hidden_dim=D)
        cached = (key, eng)
        adjacency._eval_engine = cached
    eng = cached[1]
    eng.load_state_dicts(gcn_c=gcn_c.state_dict(), gcn_gf=gcn_gf.state_dict())
    return eng
