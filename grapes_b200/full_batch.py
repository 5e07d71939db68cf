"""Full-graph training of main.py's classifier: every epoch is ONE forward of ``GCN(F, [hidden_dim, C], dropout)``
over the whole graph, main.py's classifier loss on the train rows, and one Adam step.

This is the baseline a sampler is measured against (the reference ships it as a driver of its own, ``full-batch.py``).
That file is not part of this tree, so this module restates full-graph training of main.py's classifier rather than
following it line by line: same ``Arguments`` and ``--config_file``, the loss of main.py (cross-entropy, or BCE with
logits for multi-label targets, plus ``reg_param * sum(var(logits, dim=1))`` when set), ``torch.optim.Adam(lr_gc)`` over
the classifier and, with ``--embed_nodes``, the learned node table.  The sampler fields of ``Arguments`` are ignored.

The aggregations and GEMMs, forward and backward, run on the library's kernels through the drop-in module
(:class:`grapes_b200.gcn.GCN`); loss and Adam are torch.  The gcn_norm structure of ``data.edge_index`` and its
transpose are built once per run and shared by every epoch and every evaluation.

Evaluation is full batch (``eval.evaluate(..., full_batch=True)``) whatever ``--eval_full_batch`` says: mini-batch
evaluation runs the learned sampler, and there is none here.

Without a process group the driver runs on one GPU: under ``WORLD_SIZE > 1`` it refuses, and it refuses before
allocating anything when the estimated working set (:func:`working_set_bytes`) exceeds the device's free memory.

Data parallel (``train(..., group=g)`` with more than one rank, or ``torchrun ... -m grapes_b200.full_batch``): rank r
owns the rows of its destination window of the structure (:class:`grapes_b200.gcn.ShardedGraphNorm`, windows balanced by
in-degree) and computes only those rows, forward and backward (:class:`WindowEpoch`).  Layer 2 reads Z, and the
backward's transposed aggregations read dlogits (and, with F > D, d pre) from the rows' owners over peer memory
(:class:`grapes_b200.dist.PeerRowTable`).  The partial gradients are all-gathered and added in rank order, so every rank
runs the same Adam step on the same bits and the parameters stay bit-identical across ranks.  :func:`train_emulated`
runs the same epochs for W emulated ranks in one process.  It covers the two-layer classifier with D > C and no dropout,
on a replicated fp32 or bf16 feature table; ``--embed_nodes`` is refused.

``python -m grapes_b200.full_batch --config_file ... [--flag value ...]`` prints main.py's memory and ``Acc`` lines over
``--runs``; under torchrun on rank 0 only.
"""
from __future__ import annotations

import copy
import os
from typing import List, Optional

import torch
import torch.distributed as dist
import torch.nn.functional as F

from ._lib import GrapesError, lib, ptr
from .args import Arguments, parse_cli
from .data import get_data
from .gcn import (GCN, LocalRowTable, ShardedGraphNorm, _classifier_parts, _colsum, _gemm, _gemm_into, _slab_plan,
                  row_slab_refusal)
from .graph import DeviceGraph
from .utils import _any_ctx, _stream, get_logger


def working_set_bytes(N: int, E: int, F_in: int, hidden: int, C: int, embed_nodes: bool = False, world: int = 1,
                      x_itemsize: int = 4) -> int:
    """Estimated peak device bytes of a full-graph training run: the edge list and the canonical CSR on the device, the
    structure in both directions with int64 offsets, the feature table (with ``embed_nodes`` also its gradient and two
    Adam moments), and the activations and gradients of one epoch (two [N, hidden] and three [N, F_in] and [N, C]-sized
    fp32 arrays live at the backward's peak, plus the relu output kept for the backward and a dropout mask).

    ``world`` > 1: the bytes of ONE rank of the data-parallel run, whose window holds about N / world rows and E / world
    edges in each direction: the edge list and the CSR as above, the rank's two window structures, ``dinv``, the build
    workspace and the full offsets it cuts the windows from, the table as stored (``x_itemsize`` bytes a value: 2 for
    bf16), the window's activations and gradients at the backward's peak (Y, H, d pre and its relu mask, logits, dlogits
    and dZ; with F > D the [N, D] product P on every rank and dP instead of Y) and the peer row tables (Z / dlogits, and
    d pre with F > D)."""
    C4 = (C + 3) // 4 * 4
    edges = 16 * E + (8 * (N + 1) + 4 * E)                         # edge_index on the device + canonical CSR
    if world <= 1:
        structure = 2 * (8 * (N + 1) + 4 * E) + 4 * N + 4 * N      # both directions, dinv, build workspace
        table = 4 * N * F_in * (4 if embed_nodes else 1)
        activations = 4 * N * (3 * F_in + 4 * hidden + 4 * C4) + N * hidden
        return int(edges + structure + table + activations)
    rows, wE = -(-N // world), -(-E // world)
    agg_first = F_in <= hidden
    structure = 2 * (8 * (rows + 1) + 4 * wE) + 4 * N + 4 * N + 8 * (N + 1)
    table = x_itemsize * N * F_in
    activations = rows * (4 * ((F_in if agg_first else hidden) + 2 * hidden + 3 * C4) + hidden) + \
        (0 if agg_first else 4 * N * hidden)
    tables = 4 * rows * (C4 + (0 if agg_first else hidden))
    return int(edges + structure + table + activations + tables)


def check_fits(N: int, E: int, F_in: int, hidden: int, C: int, embed_nodes: bool, device, world: int = 1,
               x_itemsize: int = 4) -> int:
    """Raise ``GrapesError`` when :func:`working_set_bytes` exceeds the free memory of ``device`` (counting what torch's
    allocator holds unused); returns the estimate."""
    need = working_set_bytes(N, E, F_in, hidden, C, embed_nodes, world, x_itemsize)
    free, _ = torch.cuda.mem_get_info(device)
    free += torch.cuda.memory_reserved(device) - torch.cuda.memory_allocated(device)
    if need > free:
        per = f" per rank of {world}" if world > 1 else ""
        raise GrapesError(f"full-graph training needs about {need} bytes ({need / 2**30:.1f} GiB) on the device{per}, "
                          f"{free} bytes ({free / 2**30:.1f} GiB) are free: N={N}, E={E}, F={F_in}, hidden={hidden}, C={C}")
    return need


def initial_model(args: Arguments, num_features: int, num_classes: int) -> GCN:
    """main.py's classifier, ``GCN(F, [hidden_dim, C], dropout)``, with weights drawn after ``torch.manual_seed(seed)``."""
    torch.manual_seed(0 if args.seed is None else args.seed)
    return GCN(num_features, [args.hidden_dim, num_classes], args.dropout)


def initial_table(args: Arguments, num_nodes: int) -> torch.Tensor:
    """main.py:95-100's learned node table, N(0, 1) [N, node_emb_dim], the host draw of ``grapes_b200.train``."""
    gen = torch.Generator().manual_seed(0 if args.seed is None else args.seed)
    return torch.empty(num_nodes, args.node_emb_dim).normal_(generator=gen)


def classifier_loss(logits: torch.Tensor, y: torch.Tensor, train_mask: torch.Tensor, reg_param: float) -> torch.Tensor:
    """main.py's ``loss_fn(logits[targets], y[targets]) + reg_param * sum(var(logits, dim=1))`` with the train rows as
    the targets and every row of the graph as the batch."""
    lg = logits[train_mask]
    if y.dim() == 1:
        loss = F.cross_entropy(lg, y[train_mask])
    else:
        loss = F.binary_cross_entropy_with_logits(lg, y[train_mask].to(lg.dtype))
    if reg_param:
        loss = loss + reg_param * torch.sum(torch.var(logits, dim=1))
    return loss


def train(args: Arguments, data=None, device: Optional[torch.device] = None, group=None):
    """Full-graph training for ``args.max_epochs`` epochs; returns ``(test_f1, mem1, mem2, mem3)`` like
    ``grapes_b200.train.train``: per epoch, the peak allocated MB, the MB the module forward reports and the MB
    allocated after the step.  ``train.last_model`` / ``train.last_table`` hold the trained classifier and, with
    ``--embed_nodes``, the learned table.  ``group``: a ``torch.distributed`` process group of more than one rank makes
    the training data parallel (see the module docstring); every rank returns the same results."""
    if group is not None and dist.get_world_size(group) > 1:
        return _train_windows(args, data, device, group=group)
    logger = get_logger()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1 or (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1):
        raise GrapesError("full-graph training without a process group runs on one GPU (WORLD_SIZE="
                          f"{world}): pass group= or run `torchrun ... -m grapes_b200.full_batch` to train data parallel")
    if not torch.cuda.is_available():
        raise GrapesError("grapes_b200 has no CPU fallback: a CUDA (sm_100a) device is required")
    if args.model_type != 'gcn':
        raise ValueError("only model_type='gcn' is wired in the reference's train() (main.py:109)")
    device = device or torch.device("cuda", torch.cuda.current_device())
    if data is None:
        path = os.path.join(os.getcwd(), 'data', args.dataset)
        data, num_features, num_classes = get_data(root=path, name=args.dataset, seed=args.seed, split_id=args.split_id)
    else:
        num_features, num_classes = data.num_features, data.num_classes
    if data.x is None and not args.embed_nodes:
        raise ValueError('Dataset does not contain node features, and embed_nodes is False. '
                         'Did you mean to run with --embed_nodes=True?')          # main.py:91-94
    F_in = args.node_emb_dim if args.embed_nodes else num_features
    need = check_fits(data.num_nodes, int(data.edge_index.shape[1]), F_in, args.hidden_dim, num_classes,
                      args.embed_nodes, device)
    logger.info(f'Full-graph training: estimated working set {need / 2**30:.2f} GiB')

    from .eval import WIDE_MIN_EDGES, _graph_norm, evaluate
    gcn_c = initial_model(args, F_in, num_classes).to(device)
    params = list(gcn_c.parameters())
    if args.embed_nodes:
        logger.info('Using learned node embeddings for features')
        x = torch.nn.Parameter(initial_table(args, data.num_nodes).to(device))
        params.append(x)
        data.x = x                                   # evaluation reads the table the optimiser updates
        data.num_features = F_in
    else:
        x = data.x.to(device).float().contiguous()
    y = data.y.to(device)
    train_mask = data.train_mask.to(device)
    optimizer = torch.optim.Adam(params, lr=args.lr_gc)

    # the structure of data.edge_index, built once: the forward direction here, the transposed one on the first backward;
    # evaluate() finds it in the graph's cache
    graph = DeviceGraph.from_edge_index(data.edge_index, data.num_nodes, device=device)
    gn = _graph_norm(graph, data, wide=int(data.edge_index.shape[1]) >= WIDE_MIN_EDGES)

    def run_eval(mask):
        res = evaluate(gcn_c, None, data, args, graph, None, 0, device, mask=mask, eval_on_cpu=False, full_batch=True)
        gcn_c.train()
        return res

    mem1, mem2, mem3 = [], [], []
    logger.info('Training')
    try:
        for epoch in range(1, args.max_epochs + 1):
            gcn_c.train()
            logits, mb = gcn_c(x, gn)
            loss = classifier_loss(logits, y, train_mask, args.reg_param)
            optimizer.zero_grad()
            loss.backward()
            optimizer.step()
            del logits
            mem1.append(torch.cuda.max_memory_allocated(device) / (1024 * 1024))
            mem2.append(mb)
            mem3.append(torch.cuda.memory_allocated(device) / (1024 * 1024))
            if (epoch + 1) % args.eval_frequency == 0:                # main.py:319
                accuracy, f1 = run_eval(data.val_mask)
                logger.info(f'epoch {epoch}: loss_c={loss.item():.6f}, valid_accuracy={accuracy:.3f}, valid_f1={f1:.3f}')
        test_accuracy, test_f1 = run_eval(data.test_mask)
        logger.info(f'test_accuracy={test_accuracy:.3f}, test_f1={test_f1:.3f}')
    finally:
        # the structure refers to the graph that caches it: drop the cache so both are freed when train() returns,
        # not at the next cyclic garbage collection
        graph._graph_norm = None
        del gn
    train.last_model = gcn_c
    train.last_table = x if args.embed_nodes else None
    return test_f1, mem1, mem2, mem3


def train_emulated(args: Arguments, data, device, world: int):
    """The data-parallel training of ``train(..., group=...)`` for ``world`` emulated ranks in one process: the windows'
    row tables are ``world`` allocations of ``device`` (:class:`grapes_b200.gcn.LocalRowTable`), every rank's phase k runs
    before any rank's phase k + 1, and the partial gradients are added in rank order as the all-gather's are, so the
    trained parameters equal those of a real ``world``-rank run bit for bit.  Evaluation is the one-process full-batch
    ``evaluate()``.  Same returns and ``train.last_model`` as :func:`train`."""
    return _train_windows(args, data, device, world=int(world))


# --------------------------------------------------------------------------------------- data-parallel full-graph epoch
class WindowEpoch:
    """One rank's share of a data-parallel full-graph training epoch of the two-layer classifier ``GCN(F, [D, C])`` with
    D > C (the classifiers of :func:`grapes_b200.gcn.row_slab_refusal`): the rank computes the rows ``lo .. hi`` of its
    window ``sgn`` only, in the phases of :meth:`phases`.  Between two phases every rank waits for all the others (the
    row tables' barrier, or, emulated, every rank's phase k before any rank's phase k + 1):

    0. layer 1 as :func:`grapes_b200.gcn.sharded_layer1` computes it (F <= D: Y = A_hat X over the window; F > D: P = X
       W1^T for all N rows), keeping Y and H = relu(. W1^T + b1) of the window; Z = H W2^T into ``z_table``;
    1. the window's logits = A_hat Z + b2 with Z read from its owners (bit-identical to the same rows of ``gcn(x,
       GraphNorm)``); main.py's loss restricted to the window -- the train-row sum over the global train-row count (for
       BCE, times C), plus ``reg_param`` times the window's sum of ``var(logits, dim=1)`` -- and its dlogits;
    2. dlogits into ``z_table`` (Z is dead: every rank has read it);
    3. dZ = A_hat^T dlogits over the transposed window, read from the owners; dW2 = dZ^T H, db2 = colsum(dlogits),
       d pre = (dZ W2) (.) (H > 0); F <= D: dW1 = d pre^T Y, db1 = colsum(d pre); F > D: d pre into ``d_table``;
    4. F > D only: dP = A_hat^T d pre read from the owners, dW1 = dP^T X over the window, db1 = colsum(d pre).

    No [N, .] array is formed except the F > D product P.  :meth:`partial` is the flat partial gradient (parameters in
    ``gcn.named_parameters()`` order) followed by the window's loss; :func:`sum_in_rank_order` of every rank's partial is
    the epoch's gradient and loss."""

    SLAB_ROWS = 1 << 20           # rows per launch, the whole-graph launch shape of the row-slab kernels

    def __init__(self, gcn: GCN, x: torch.Tensor, sgn: ShardedGraphNorm, z_table, y: torch.Tensor,
                 train_mask: torch.Tensor, n_train: int, reg_param: float = 0., d_table=None):
        w1, b1, w2, b2, D, C, C4 = _classifier_parts(gcn, x)
        F_in = x.shape[1]
        if z_table.ld != C4 or z_table.rows.shape[0] < sgn.rows:
            raise GrapesError(f"row table of pitch {z_table.ld} x {z_table.rows.shape[0]} rows; the window needs "
                              f"{C4} x {sgn.rows}")
        if F_in > D and (d_table is None or d_table.ld != D or d_table.rows.shape[0] < sgn.rows):
            raise GrapesError(f"F = {F_in} > D = {D}: the backward needs a d pre row table of pitch {D} x {sgn.rows} rows")
        self.gcn, self.x, self.sgn, self.z_table, self.d_table = gcn, x, sgn, z_table, d_table
        self.D, self.C, self.C4, self.agg_first = D, C, C4, F_in <= D
        lo, hi = sgn.lo, sgn.hi
        self.y, self.mask = y[lo:hi], train_mask[lo:hi]
        self.n_train, self.reg_param = int(n_train), float(reg_param)
        self.R = max(1, min(self.SLAB_ROWS, sgn.rows))
        self.starts, self.slabs = _slab_plan(lo, hi, self.R, sgn.dinv.device)

    def phases(self):
        return [self._layer1, self._layer2_loss, self._publish_dlogits, self._backward2] + \
            ([] if self.agg_first else [self._backward1])

    def _slab_views(self):
        lo = self.sgn.lo
        for i, r0 in enumerate(self.starts):
            yield self.slabs[i], r0 - lo, min(self.R, self.sgn.hi - r0)

    def _layer1(self):
        w1, b1, w2, b2, D, C, C4 = _classifier_parts(self.gcn, self.x)
        self.w2, self.b2 = w2, b2
        x, sgn, rows = self.x, self.sgn, self.sgn.rows
        dev = sgn.dinv.device
        N, F_in = x.shape
        self.Y = torch.empty((rows, F_in), dtype=torch.float32, device=dev) if self.agg_first else None
        self.H = torch.empty((rows, D), dtype=torch.float32, device=dev)
        if rows == 0:
            return
        if self.agg_first:
            for slab, a, n in self._slab_views():
                sgn.aggregate_rows(x, slab, n, self.Y[a:])
                _gemm_into(self.Y[a:], F_in, w1, F_in, self.H[a:], D, n, D, F_in, bias=b1)
        else:                     # the sources of the window may be any rows: P for all N, as the streamed forward
            P = torch.empty((N, D), dtype=torch.float32, device=dev)
            for r0 in range(0, N, self.SLAB_ROWS):
                n = min(self.SLAB_ROWS, N - r0)
                xs = x[r0:r0 + n] if x.dtype == torch.float32 else x[r0:r0 + n].float()
                _gemm_into(xs, xs.stride(0), w1, F_in, P[r0:], D, n, D, F_in)
            for slab, a, n in self._slab_views():
                sgn.aggregate_rows(P, slab, n, self.H[a:], bias=b1)
            del P
        torch.relu_(self.H)
        for slab, a, n in self._slab_views():
            _gemm_into(self.H[a:], D, w2, D, self.z_table.rows[a:], C4, n, C, D)

    def _layer2_loss(self):
        sgn, C, C4 = self.sgn, self.C, self.C4
        out = torch.empty((sgn.rows, C4), dtype=torch.float32, device=sgn.dinv.device)
        for slab, a, n in self._slab_views():
            sgn.aggregate_rows_peer(self.z_table, slab, n, out[a:], bias=self.b2)
        self.logits = out[:, :C]
        lg = self.logits.detach().clone().requires_grad_(True)
        with torch.enable_grad():
            loss = window_loss(lg, self.y, self.mask, self.n_train, self.reg_param)
            loss.backward()
        self.loss, self.dlogits = loss.detach().reshape(1), lg.grad.contiguous()

    def _publish_dlogits(self):
        self.z_table.rows[:self.sgn.rows, :self.C].copy_(self.dlogits)

    def _backward2(self):
        sgn, D, C, C4, rows = self.sgn, self.D, self.C, self.C4, self.sgn.rows
        dev = sgn.dinv.device
        dZ = torch.empty((rows, C4), dtype=torch.float32, device=dev)
        for slab, a, n in self._slab_views():
            sgn.aggregate_rows_peer(self.z_table, slab, n, dZ[a:], transpose=True, F=C)
        self.dW2 = _gemm_tn_ld(dZ, C4, self.H, D, rows, C, D)
        self.db2 = _colsum(self.dlogits)
        self.dlogits = None
        dpre = _gemm(1, dZ, C4, self.w2, D, rows, D, C)                     # dZ W2
        del dZ
        dpre.masked_fill_(self.H <= 0, 0.)                                    # relu'
        self.db1 = _colsum(dpre)
        if self.agg_first:
            self.dW1 = _gemm_tn_ld(dpre, D, self.Y, self.Y.shape[1], rows, D, self.Y.shape[1])
            self.Y = self.H = None
        else:
            self.d_table.rows[:rows].copy_(dpre)
            self.H = None
        del dpre

    def _backward1(self):
        sgn, D, rows = self.sgn, self.D, self.sgn.rows
        F_in = self.x.shape[1]
        dP = torch.empty((rows, D), dtype=torch.float32, device=sgn.dinv.device)
        for slab, a, n in self._slab_views():
            sgn.aggregate_rows_peer(self.d_table, slab, n, dP[a:], transpose=True)
        xw = self.x[sgn.lo:sgn.hi]
        xw = xw if xw.dtype == torch.float32 else xw.float()
        self.dW1 = _gemm_tn_ld(dP, D, xw, F_in, rows, D, F_in)

    def partial(self) -> torch.Tensor:
        """This rank's flat partial gradient, parameters in ``gcn.named_parameters()`` order, then the window's loss."""
        g = {"gcn_layers.0.lin.weight": self.dW1, "gcn_layers.0.bias": self.db1,
             "gcn_layers.1.lin.weight": self.dW2, "gcn_layers.1.bias": self.db2}
        return torch.cat([g[n].reshape(-1) for n, _ in self.gcn.named_parameters()] + [self.loss])


def _gemm_tn_ld(A, lda: int, B, ldb: int, R: int, M: int, N: int) -> torch.Tensor:
    """A^T B [M, N] over R rows of A (pitch lda) and B (pitch ldb): ``grapes_gemm_tn``."""
    out = torch.zeros((M, N), dtype=torch.float32, device=A.device)
    if R > 0:
        lib().grapes_gemm_tn(_any_ctx(A.device).ctx, ptr(A), lda, ptr(B), ldb, None, R, M, N, 1.0, 0, ptr(out), _stream())
    return out


def window_loss(logits: torch.Tensor, y: torch.Tensor, train_mask: torch.Tensor, n_train: int,
                reg_param: float) -> torch.Tensor:
    """The window's share of :func:`classifier_loss`: the sum of the per-row loss over the window's train rows divided
    by the train-row count of the whole graph (times C for the element mean of BCE), plus ``reg_param`` times the sum of
    ``var(logits, dim=1)`` over the window's rows.  The shares of all windows add up to :func:`classifier_loss`."""
    lg = logits[train_mask]
    if y.dim() == 1:
        loss = F.cross_entropy(lg, y[train_mask], reduction="sum") / n_train
    else:
        loss = F.binary_cross_entropy_with_logits(lg, y[train_mask].to(lg.dtype), reduction="sum") / \
            (n_train * logits.shape[1])
    if reg_param and logits.shape[0] > 0:
        loss = loss + reg_param * torch.sum(torch.var(logits, dim=1))
    return loss


def sum_in_rank_order(parts: List[torch.Tensor]) -> torch.Tensor:
    """parts[0] + parts[1] + ... in that order (a new tensor): the reduction both the all-gathered and the emulated
    partial gradients take, so the result does not depend on how the ranks ran."""
    total = parts[0].clone()
    for p in parts[1:]:
        total += p
    return total


def run_epoch(epoch: WindowEpoch, group) -> torch.Tensor:
    """One epoch of this rank over ``group``: the phases with a barrier after each, then the all-gather of the partial
    gradients summed in rank order.  Returns the flat gradient and loss, the same bits on every rank."""
    for phase in epoch.phases():
        phase()
        epoch.z_table.barrier()
    mine = epoch.partial()
    parts = [torch.empty_like(mine) for _ in range(dist.get_world_size(group))]
    dist.all_gather(parts, mine, group=group)
    return sum_in_rank_order(parts)


def run_epoch_emulated(epochs: List[WindowEpoch]) -> torch.Tensor:
    """:func:`run_epoch` for emulated ranks in one process: every rank's phase k before any rank's phase k + 1."""
    for k in range(len(epochs[0].phases())):
        for e in epochs:
            e.phases()[k]()
    return sum_in_rank_order([e.partial() for e in epochs])


def _set_grads(gcn: GCN, flat: torch.Tensor) -> torch.Tensor:
    """p.grad of every parameter from the flat gradient; returns the loss at its end."""
    a = 0
    for _, p in gcn.named_parameters():
        p.grad = flat[a:a + p.numel()].view_as(p).clone()
        a += p.numel()
    return flat[a]


def data_parallel_refusal(args: Arguments, data, num_classes: int) -> Optional[str]:
    """Why the data-parallel driver does not train this configuration, or None: decided from the arguments and the
    table's type alone, so every rank refuses alike and before allocating anything."""
    from .dist import ShardedFeatures
    if args.embed_nodes:
        return "--embed_nodes is not supported by data-parallel full-graph training"
    if args.dropout > 0:
        return "--dropout > 0 is not supported by data-parallel full-graph training"
    if isinstance(data.x, ShardedFeatures):
        return "data-parallel full-graph training reads a replicated feature table, not a sharded one"
    if data.x is None:
        return "data-parallel full-graph training needs node features (data.x)"
    why = row_slab_refusal(GCN(data.x.shape[1], [args.hidden_dim, num_classes]), data.x)
    return None if why is None else f"data-parallel full-graph training: {why}"


def _peer_table(rows: int, ld: int, device, group):
    """A :class:`grapes_b200.dist.PeerRowTable` mapped on every rank of ``group``, or ``GrapesError`` on every rank."""
    from .dist import PeerRowTable, ranks_agree
    table, why = None, ""
    try:
        table = PeerRowTable(rows, ld, device, group)
    except Exception as exc:                            # noqa: BLE001 -- agreed below and raised on every rank
        why = f"{type(exc).__name__}: {exc}"
    if ranks_agree(table is not None, device, group):
        try:
            table.rendezvous()
        except Exception as exc:                        # noqa: BLE001
            why, table = f"{type(exc).__name__}: {exc}", None
        if not ranks_agree(table is not None, device, group):
            table = None
    else:
        table = None
    if table is None:
        raise GrapesError("data-parallel full-graph training: peer row table could not be mapped " +
                          (f"on this rank ({why})" if why else "on another rank"))
    return table


def _train_windows(args: Arguments, data, device, group=None, world: int = 1):
    """The data-parallel driver of :func:`train` (``group``) and :func:`train_emulated` (``world`` emulated ranks)."""
    from .dist import ranks_agree
    from .eval import _sharded_eval, evaluate
    logger = get_logger()
    if not torch.cuda.is_available():
        raise GrapesError("grapes_b200 has no CPU fallback: a CUDA (sm_100a) device is required")
    if args.model_type != 'gcn':
        raise ValueError("only model_type='gcn' is wired in the reference's train() (main.py:109)")
    emulated = group is None
    if not emulated:
        world, rank = dist.get_world_size(group), dist.get_rank(group)
    device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    if data is None:
        path = os.path.join(os.getcwd(), 'data', args.dataset)
        data, num_features, num_classes = get_data(root=path, name=args.dataset, seed=args.seed, split_id=args.split_id)
    else:
        num_features, num_classes = data.num_features, data.num_classes
    why = data_parallel_refusal(args, data, num_classes)
    if why is not None:
        raise GrapesError(why)
    N, E, F_in = data.num_nodes, int(data.edge_index.shape[1]), int(data.x.shape[1])
    fits, need = True, 0
    try:
        need = check_fits(N, E, F_in, args.hidden_dim, num_classes, False, device, world, data.x.element_size())
    except GrapesError:
        if emulated:
            raise
        fits = False
    if not emulated and not ranks_agree(fits, device, group):
        raise GrapesError("data-parallel full-graph training: the estimated working set of a rank "
                          f"({working_set_bytes(N, E, F_in, args.hidden_dim, num_classes, False, world, data.x.element_size())}"
                          " bytes) exceeds the free memory of this rank or another")
    logger.info(f'Data-parallel full-graph training over {world} ranks: estimated working set {need / 2**30:.2f} GiB '
                'per rank')

    gcn_c = initial_model(args, F_in, num_classes).to(device)
    D, C = args.hidden_dim, num_classes
    C4 = (C + 3) // 4 * 4
    x = data.x.to(device).contiguous()                  # as stored: the row kernels widen bf16 on read
    y = data.y.to(device)
    train_mask = data.train_mask.to(device)
    n_train = int(train_mask.sum())
    optimizer = torch.optim.Adam(gcn_c.parameters(), lr=args.lr_gc)
    ev_data = copy.copy(data)
    ev_data.x = x                                       # evaluation reads the device table, not a second copy

    graph = DeviceGraph.from_edge_index(data.edge_index, N, device=device)
    try:
        if emulated:
            sgns = [ShardedGraphNorm(graph, world, r, edge_index=data.edge_index) for r in range(world)]
            rows = max(s.rows for s in sgns)
            z_tables = LocalRowTable.make(world, rows, C4, device)
            d_tables = LocalRowTable.make(world, rows, D, device) if F_in > D else [None] * world
        else:
            # the window structure and Z table of the data-parallel evaluation, cached on the graph: evaluate() reuses them
            sgn, z_table, _ = _sharded_eval(graph, data, group, C4, device, fallback=False)
            if z_table is None:
                raise GrapesError("data-parallel full-graph training: window structure or peer-mapped row table "
                                  f"unavailable ({graph._sharded_eval_failure})")
            rows = max(sgn.bounds[r + 1] - sgn.bounds[r] for r in range(world))
            sgns, z_tables = [sgn], [z_table]
            d_tables = [_peer_table(rows, D, device, group) if F_in > D else None]
        for s in sgns:
            s.build_transposed()
        epochs = [WindowEpoch(gcn_c, x, s, zt, y, train_mask, n_train, args.reg_param, dt)
                  for s, zt, dt in zip(sgns, z_tables, d_tables)]

        def run_eval(mask):
            res = evaluate(gcn_c, None, ev_data, args, graph, None, 0, device, mask=mask, eval_on_cpu=False,
                           full_batch=True, group=group)
            gcn_c.train()
            return res

        mem1, mem2, mem3 = [], [], []
        logger.info('Training')
        for epoch in range(1, args.max_epochs + 1):
            gcn_c.train()
            flat = run_epoch_emulated(epochs) if emulated else run_epoch(epochs[0], group)
            mem2.append(torch.cuda.memory_allocated(device) / (1024 * 1024))
            loss = _set_grads(gcn_c, flat)
            optimizer.step()
            mem1.append(torch.cuda.max_memory_allocated(device) / (1024 * 1024))
            mem3.append(torch.cuda.memory_allocated(device) / (1024 * 1024))
            if (epoch + 1) % args.eval_frequency == 0:                # main.py:319
                accuracy, f1 = run_eval(data.val_mask)
                logger.info(f'epoch {epoch}: loss_c={loss.item():.6f}, valid_accuracy={accuracy:.3f}, valid_f1={f1:.3f}')
        test_accuracy, test_f1 = run_eval(data.test_mask)
        logger.info(f'test_accuracy={test_accuracy:.3f}, test_f1={test_f1:.3f}')
    finally:
        # the structures and tables refer to the graph that caches them: drop them when train() returns
        graph._graph_norm = None
        graph._sharded_eval, graph._sharded_eval_p = None, None
        epochs = sgns = z_tables = d_tables = None
    train.last_model = gcn_c
    train.last_table = None
    return test_f1, mem1, mem2, mem3


def main(argv=None):
    from .main import report
    args = parse_cli(argv)
    group = None
    if int(os.environ.get("WORLD_SIZE", "1")) > 1:
        if not dist.is_initialized():
            local = int(os.environ.get("LOCAL_RANK", "0"))
            torch.cuda.set_device(local)
            dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        group = dist.group.WORLD
    results = torch.empty(args.runs)
    mem1, mem2, mem3 = [], [], []
    for r in range(args.runs):
        test_f1, m1, m2, m3 = train(args, group=group)
        results[r] = test_f1
        mem1.extend(m1); mem2.extend(m2); mem3.extend(m3)
    if group is None or dist.get_rank(group) == 0:
        report(results, mem1, mem2, mem3)


if __name__ == "__main__":
    main()
