"""``train(args)`` with the reference's contract (/root/reference/main.py:57-364): same ``Arguments``,
same epoch / batch order (sequential, un-shuffled batches of ``train_idx``, last batch partial,
main.py:125-126), same return tuple ``(test_f1, mem_point1, mem_point2, mem_point3)``; the batch body runs
on :class:`grapes_b200.engine.GrapesEngine` instead of scipy + PyG.
"""
from __future__ import annotations

import os
from typing import Optional

import torch

from ._lib import GrapesError
from .args import Arguments
from .data import get_data
from .engine import GrapesEngine, STAT_NAMES
from .gcn import GCN
from .graph import DeviceGraph
from .utils import get_logger


def evaluate(engine: GrapesEngine, data, mask: torch.Tensor, full_batch: bool = True, args=None, graph=None, group=None):
    """The reference's two evaluation modes (/root/reference/eval.py:47-70 full-batch, :71-163 mini-batch) on the
    device, with the engine's current weights loaded into drop-in ``GCN`` modules (grapes_b200/eval.py); data parallel
    over ``group`` when it has more than one rank.  Reads the engine's feature table when it is sharded."""
    from .eval import evaluate as _evaluate
    dev = engine.device
    sd = engine.state_dicts()
    gcn_c = GCN(engine.F, [engine.D, engine.C]).to(dev)
    gcn_c.load_state_dict(sd["gcn_c"])
    gcn_gf = GCN(engine.Fp, [engine.D, 1]).to(dev)
    gcn_gf.load_state_dict(sd["gcn_gf"])
    graph = graph or engine.g
    loader = None
    if not full_batch:
        idx = mask.nonzero().squeeze(1)
        loader = [(b,) for b in torch.split(idx, engine.B)]         # DataLoader(TensorDataset(idx), batch_size=args.batch_size) main.py:127-132
    ns = args if args is not None else type("A", (), dict(sampling_hops=engine.H, num_samples=engine.k,
                                                          use_indicators=engine.use_ind))()
    return _evaluate(gcn_c, gcn_gf, data, ns, graph, None, engine.num_ind, dev, mask=mask, eval_on_cpu=False,
                     loader=loader, full_batch=full_batch, engine=None if full_batch else engine, group=group,
                     features=engine.features)


def train(args: Arguments, data=None, device: Optional[torch.device] = None, use_cuda_graph: bool = True,
          max_batches: Optional[int] = None, exchange: str = "peer", step_log=None, shard_eval: bool = True, *,
          shard_features: bool = False, shard_embeddings: bool = False, checkpoint_dir: Optional[str] = None,
          checkpoint_every: int = 0, resume: bool = False):
    """``train(args)`` of the reference (main.py:57-364).  Under ``torchrun`` (WORLD_SIZE > 1, or an initialised
    ``torch.distributed`` group) it is data parallel: every rank holds a replica of the graph and features, batch ``i`` of
    the un-shuffled loader goes to rank ``i mod W`` (``dist.shard_batches``), and the engine exchanges the gradient and
    applies both optimisers inside its step, so all ranks hold the same weights (BASELINE.json north_star).
    ``step_log(dict)`` (optional) receives what main.py:293-311 sends to wandb for every batch -- batch losses, log_z,
    -log_probs and the per-hop sampler statistics ``{min_prob,max_prob,mean_entropy,std_entropy}_{hop}`` -- one step
    behind, read from pinned host memory (no device stall).  ``shard_eval`` (data parallel only): every evaluation is
    split between the ranks (``eval.evaluate(..., group=...)``, the same scores); False makes every rank evaluate the whole
    mask, as one process does.

    ``shard_features`` (data parallel only; no effect with one process): the feature table is sharded by rows across the
    ranks (:class:`grapes_b200.dist.ShardedFeatures`) instead of replicated, each rank holding 1/W of it and gathering
    the other rows over NVLink peer memory, with bit-identical results.  For tables that do not fit one GPU: ``data.x``
    may stay on the host (memory-mapped or not) and is never moved to one device whole.  Not with ``--embed_nodes``, and
    full-batch evaluation needs ``shard_eval``.

    ``shard_embeddings`` (data parallel with ``--embed_nodes`` only; no effect with one process): the learned table and
    its two Adam moments are sharded by rows across the ranks (:class:`grapes_b200.dist.ShardedEmbedding`); each rank
    updates only its rows and reads the others from their owners, with results bit-identical to the replicated learned
    table.  Full-batch evaluation needs ``shard_eval``.  The initial table is still drawn whole on the host of every
    process (N x node_emb_dim floats) before each rank keeps its rows, unless the run resumes from a checkpoint.

    ``checkpoint_dir``: a checkpoint (:mod:`grapes_b200.checkpoint`) is written there at the end of every epoch, after
    that epoch's evaluation, and with ``checkpoint_every = n > 0`` also after every n steps of the rank.  ``resume``:
    the run continues from the directory's latest checkpoint (its epoch, batch, loss accumulators and every device
    state), bit-identical to a run that never stopped; without one it starts fresh.  A resumed ``--embed_nodes`` run
    reads the learned table from the checkpoint and draws no initial table.  The memory points returned cover only
    the steps this process ran."""
    logger = get_logger()
    if checkpoint_every < 0 or (checkpoint_every and checkpoint_dir is None) or (resume and checkpoint_dir is None):
        raise GrapesError("checkpoint_every > 0 and resume need checkpoint_dir")
    if shard_features and args.embed_nodes:
        raise GrapesError("shard_features with --embed_nodes: the learned table's optimiser is not sharded; "
                          "replicate the table (shard_features=False)")
    if shard_embeddings and not args.embed_nodes:
        raise GrapesError("shard_embeddings shards the learned table of --embed_nodes; to shard a given feature table "
                          "use shard_features=True")
    if shard_embeddings and args.eval_full_batch and not shard_eval:
        raise GrapesError("shard_embeddings with full-batch evaluation needs shard_eval=True: no rank holds the whole "
                          "table to evaluate alone")
    if shard_features and args.eval_full_batch and not shard_eval:
        raise GrapesError("shard_features with full-batch evaluation needs shard_eval=True: no rank holds the whole "
                          "table to evaluate alone")
    if not torch.cuda.is_available():
        raise GrapesError("grapes_b200 has no CPU fallback: a CUDA (sm_100a) device is required")
    import torch.distributed as dist
    from .dist import shard_batches
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world > 1 and not dist.is_initialized():
        local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    world = dist.get_world_size() if dist.is_initialized() else 1
    rank = dist.get_rank() if dist.is_initialized() else 0
    device = device or torch.device("cuda", torch.cuda.current_device())
    if data is None:
        path = os.path.join(os.getcwd(), 'data', args.dataset)
        data, num_features, num_classes = get_data(root=path, name=args.dataset, seed=args.seed, split_id=args.split_id)
    else:
        num_features, num_classes = data.num_features, data.num_classes
    from .checkpoint import latest, load, save, table_source
    resume_from = latest(checkpoint_dir) if resume else None
    if resume and resume_from is None:
        logger.info(f'No checkpoint in {checkpoint_dir}: starting fresh')
    if args.embed_nodes or data.x is None:
        if not args.embed_nodes:
            raise ValueError('Dataset does not contain node features, and embed_nodes is False. '
                             'Did you mean to run with --embed_nodes=True?')          # main.py:91-94
        logger.info('Using learned node embeddings for features')
        if resume_from is not None:
            # the table and its moments come from the checkpoint (load() below): no initial draw
            if shard_embeddings and world > 1:
                data.x = table_source(resume_from)[0]    # memory-mapped [N, F]: each rank fills its rows from it
            else:
                data.x = torch.empty(data.num_nodes, args.node_emb_dim, device=device)
        else:
            # main.py:95-100: embeddings = nn.Parameter(FloatTensor(N, node_emb_dim).normal_()), appended to optimizer_c.
            # Here the table lives in HBM and the engine's optimiser launch updates it in place (grapes_adam_embed); under
            # torchrun it is replicated and every rank applies the mean of the ranks' row-sparse gradients.
            gen = torch.Generator().manual_seed(0 if args.seed is None else args.seed)
            data.x = torch.empty(data.num_nodes, args.node_emb_dim).normal_(generator=gen)
            if not (shard_embeddings and world > 1):
                data.x = data.x.to(device)       # a sharded table is filled rank by rank from the host draw
        data.num_features = num_features = args.node_emb_dim
    if args.model_type != 'gcn':
        raise ValueError("only model_type='gcn' is wired in the reference's train() (main.py:109)")

    # frontier capacity of the library context: a batch expands at most (B + k) rows of at most max_deg entries
    graph = DeviceGraph.from_edge_index(data.edge_index, data.num_nodes, device=device)
    deg = graph.indptr[1:] - graph.indptr[:-1]
    need = min(graph.nnz, (args.batch_size + args.num_samples) * max(int(deg.max().item()) if graph.nnz else 1, 1), 1 << 26)
    if need + args.batch_size + args.num_samples > graph.max_frontier:
        graph = DeviceGraph(graph.indptr, graph.indices, data.num_nodes,
                            max_frontier=need + args.batch_size + args.num_samples)
    sharded_table = shard_embeddings and world > 1
    if sharded_table:
        from .dist import ShardedEmbedding
        x_dev = ShardedEmbedding(data.x, device)     # collective; every rank fills its rows from the same draw
    elif shard_features and world > 1:
        from .dist import ShardedFeatures
        x_dev = ShardedFeatures(data.x, device)      # collective; raises on every rank when any rank cannot map it
    else:
        x_dev = data.x.to(device).contiguous()
    if args.embed_nodes:
        data.x = x_dev                       # evaluation reads the table the optimiser updates
    engine = GrapesEngine(graph, x_dev, data.y.to(device), num_classes=num_classes, embed_nodes=args.embed_nodes,
                          batch_size=args.batch_size, num_samples=args.num_samples, sampling_hops=args.sampling_hops,
                          use_indicators=args.use_indicators, hidden_dim=args.hidden_dim, lr_gc=args.lr_gc,
                          lr_gf=args.lr_gf, loss_coef=args.loss_coef, log_z_init=args.log_z_init,
                          reg_param=args.reg_param, random_sampling=args.random_sampling,
                          reinforce_baseline=args.reinforce_baseline, seed=0 if args.seed is None else args.seed,
                          dropout=args.dropout)                # gcn_c only (main.py:107-112); evaluation never drops
    if world > 1:
        engine.enable_data_parallel(exchange=exchange)
    eval_group = dist.group.WORLD if world > 1 and shard_eval else None
    train_idx = data.train_mask.nonzero().squeeze(1).to(device)
    batches = [b.to(torch.int32).contiguous() for b in torch.split(train_idx, args.batch_size)]   # DataLoader(TensorDataset(train_idx), batch_size)
    if max_batches is not None:
        batches = batches[:max_batches]
    if world > 1:
        batches = [batches[i] for i in shard_batches(len(batches), rank, world)]

    # every step's losses, flag bits and per-hop sampler statistics are copied to pinned host memory and read ONE STEP
    # BEHIND (the reference reads loss.item() every batch, main.py:269,291: a device stall here)
    nread = engine.scal_stats.numel()
    host = [torch.zeros(nread, dtype=torch.float32).pin_memory() for _ in range(2)]
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    state = {"pending": None, "acc_c": 0.0, "acc_gfn": 0.0, "last": None}
    start_epoch, start_batch, step_no = 1, 0, 0
    if resume_from is not None:
        loop = load(engine, resume_from, args=args)
        state.update(acc_c=loop["acc_c"], acc_gfn=loop["acc_gfn"], last=loop["last"])
        start_epoch, start_batch, step_no = loop["epoch"], loop["batch"], loop["step"]
        if start_batch >= len(batches):                  # saved at the end of its epoch
            start_epoch, start_batch = start_epoch + 1, 0
        logger.info(f'Resuming from {resume_from}: epoch {start_epoch}, batch {start_batch}, step {step_no}')

    def collect():
        j = state["pending"]
        if j is None:
            return
        ready[j % 2].synchronize()
        h = host[j % 2]
        engine.raise_on_flags(int(h[15]))                 # frontier overflow / failed exchange of THAT step: stop now
        nb = max(len(batches), 1)
        state["acc_c"] += float(h[0]) / nb
        state["acc_gfn"] += float(h[4]) / nb
        log = {'batch_loss_gfn': float(h[4]), 'batch_loss_c': float(h[0]), 'log_z': float(h[3]),
               '-log_probs': -float(h[1])}
        for hop in range(engine.H):                       # main.py:304-308
            for i, key in enumerate(STAT_NAMES):
                log[f"{key}_{hop}"] = float(h[16 + 4 * hop + i])
        state["last"] = log
        if step_log is not None:
            step_log(log)
        state["pending"] = None

    def sync_ranks():
        # a sharded learned table: every rank's last table step is applied before any rank's evaluation reads its rows
        if sharded_table:
            from .dist import ranks_agree
            torch.cuda.synchronize(device)
            ranks_agree(True, device)

    def checkpoint(epoch, done):
        collect()                                         # the step log is complete up to the checkpoint
        save(engine, checkpoint_dir, dict(epoch=epoch, batch=done, step=step_no, acc_c=state["acc_c"],
                                          acc_gfn=state["acc_gfn"], last=state["last"]), args=args)

    mem1, mem2, mem3 = [], [], []
    logger.info('Training')
    test_f1 = 0.0
    for epoch in range(start_epoch, args.max_epochs + 1):
        first = start_batch if epoch == start_epoch else 0
        if first == 0:
            state["acc_c"] = state["acc_gfn"] = 0.0
        for bi in range(first, len(batches)):
            batch = batches[bi]
            # the next batch's reset + hop-0 front end is enqueued next to this step's classifier tail
            engine.step(batch, use_graph=use_cuda_graph, next_targets=batches[bi + 1] if bi + 1 < len(batches) else None)
            host[step_no % 2].copy_(engine.scal_stats, non_blocking=True)
            ready[step_no % 2].record()
            collect()
            state["pending"] = step_no
            step_no += 1
            # main.py:265,284-285: memory points.  Every buffer of the step is allocated once, so the three points see
            # the same allocator state: point 1 = peak, point 2 (what GCN.forward reports) and point 3 = current
            mb = torch.cuda.memory_allocated() / (1024 * 1024)
            if not args.random_sampling:
                mem1.append(torch.cuda.max_memory_allocated() / (1024 * 1024)); mem2.append(mb)
            mem3.append(mb)
            # the last batch of an epoch is checkpointed after the epoch's evaluation instead
            if checkpoint_every and step_no % checkpoint_every == 0 and bi + 1 < len(batches):
                checkpoint(epoch, bi + 1)
        collect()
        engine.check_overflow()
        if (epoch + 1) % args.eval_frequency == 0:                # main.py:319
            sync_ranks()
            accuracy, f1 = evaluate(engine, data, data.val_mask, full_batch=args.eval_full_batch, args=args,
                                    group=eval_group)
            logger.info(f'loss_gfn={state["acc_gfn"]:.6f}, loss_c={state["acc_c"]:.6f}, '
                        f'valid_accuracy={accuracy:.3f}, valid_f1={f1:.3f}')
        if checkpoint_dir is not None:
            checkpoint(epoch, len(batches))
    sync_ranks()
    test_accuracy, test_f1 = evaluate(engine, data, data.test_mask, full_batch=args.eval_full_batch, args=args,
                                      group=eval_group)
    logger.info(f'test_accuracy={test_accuracy:.3f}, test_f1={test_f1:.3f}')
    train.last_engine = engine
    train.last_log = state["last"]
    return test_f1, mem1, mem2, mem3
