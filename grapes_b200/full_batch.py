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

Single GPU only: under ``WORLD_SIZE > 1`` the driver refuses, and it refuses before allocating anything when the
estimated working set (:func:`working_set_bytes`) exceeds the device's free memory.

``python -m grapes_b200.full_batch --config_file ... [--flag value ...]`` prints main.py's memory and ``Acc`` lines over
``--runs``.
"""
from __future__ import annotations

import os
from typing import Optional

import torch
import torch.nn.functional as F

from ._lib import GrapesError
from .args import Arguments, parse_cli
from .data import get_data
from .gcn import GCN
from .graph import DeviceGraph
from .utils import get_logger


def working_set_bytes(N: int, E: int, F_in: int, hidden: int, C: int, embed_nodes: bool = False) -> int:
    """Estimated peak device bytes of a full-graph training run: the edge list and the canonical CSR on the device, the
    structure in both directions with int64 offsets, the feature table (with ``embed_nodes`` also its gradient and two
    Adam moments), and the activations and gradients of one epoch (two [N, hidden] and three [N, F_in] and [N, C]-sized
    fp32 arrays live at the backward's peak, plus the relu output kept for the backward and a dropout mask)."""
    C4 = (C + 3) // 4 * 4
    edges = 16 * E + (8 * (N + 1) + 4 * E)                         # edge_index on the device + canonical CSR
    structure = 2 * (8 * (N + 1) + 4 * E) + 4 * N + 4 * N          # both directions, dinv, build workspace
    table = 4 * N * F_in * (4 if embed_nodes else 1)
    activations = 4 * N * (3 * F_in + 4 * hidden + 4 * C4) + N * hidden
    return int(edges + structure + table + activations)


def check_fits(N: int, E: int, F_in: int, hidden: int, C: int, embed_nodes: bool, device) -> int:
    """Raise ``GrapesError`` when :func:`working_set_bytes` exceeds the free memory of ``device`` (counting what torch's
    allocator holds unused); returns the estimate."""
    need = working_set_bytes(N, E, F_in, hidden, C, embed_nodes)
    free, _ = torch.cuda.mem_get_info(device)
    free += torch.cuda.memory_reserved(device) - torch.cuda.memory_allocated(device)
    if need > free:
        raise GrapesError(f"full-graph training needs about {need} bytes ({need / 2**30:.1f} GiB) on the device, "
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


def train(args: Arguments, data=None, device: Optional[torch.device] = None):
    """Full-graph training for ``args.max_epochs`` epochs; returns ``(test_f1, mem1, mem2, mem3)`` like
    ``grapes_b200.train.train``: per epoch, the peak allocated MB, the MB the module forward reports and the MB
    allocated after the step.  ``train.last_model`` / ``train.last_table`` hold the trained classifier and, with
    ``--embed_nodes``, the learned table."""
    logger = get_logger()
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1 or (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1):
        raise GrapesError("full-graph training runs on one GPU: data-parallel full-graph training is not supported "
                          f"(WORLD_SIZE={world})")
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


def main(argv=None):
    from .main import report
    args = parse_cli(argv)
    results = torch.empty(args.runs)
    mem1, mem2, mem3 = [], [], []
    for r in range(args.runs):
        test_f1, m1, m2, m3 = train(args)
        results[r] = test_f1
        mem1.extend(m1); mem2.extend(m2); mem3.extend(m3)
    report(results, mem1, mem2, mem3)


if __name__ == "__main__":
    main()
