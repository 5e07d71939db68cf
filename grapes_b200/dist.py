"""Data-parallel plumbing (new work defined by BASELINE.json; the reference is single-process).

One process per GPU, CSR + features replicated, target-node batches sharded by index, and ONE collective per
step: the mean all-reduce of the flat gradient buffer (gcn_c | gcn_gf | gcn_z; 91 k floats on products-shape).
``loss_c.detach()`` inside the GFlowNet loss is rank-local (main.py:274), so nothing else is exchanged.
The trajectory-balance loss is the square of a per-batch scalar, so W-rank data parallelism equals averaging
W per-batch gradients -- not one W x B batch (SURVEY.md section 7.2)."""
from __future__ import annotations

from typing import List, Tuple

import torch
import torch.distributed as dist


def shard_batches(num_batches: int, rank: int, world: int) -> List[int]:
    """Batch i of the un-shuffled loader (main.py:125-126) goes to rank i mod W; every rank runs the same
    number of steps (the tail that does not fill a full round is dropped so no rank waits at the all-reduce)."""
    rounds = num_batches // world
    return [r * world + rank for r in range(rounds)]


def allreduce_mean_(flat: torch.Tensor) -> torch.Tensor:
    """In-place mean over ranks of a flat buffer (NCCL: one ReduceOp.AVG call; gloo: SUM then divide)."""
    if not dist.is_initialized() or dist.get_world_size() == 1:
        return flat
    if dist.get_backend() == "nccl":
        dist.all_reduce(flat, op=dist.ReduceOp.AVG)
    else:
        dist.all_reduce(flat, op=dist.ReduceOp.SUM)
        flat.div_(dist.get_world_size())
    return flat


def ranks_agree(ok: bool, device, group=None) -> bool:
    """True iff EVERY rank of ``group`` passed ok=True (all-reduce MIN of a flag; also a synchronisation point of the
    ranks).  Used where a rank-local decision would deadlock the group: whether the peer-memory exchange could be set up
    (``GrapesEngine.enable_data_parallel``)."""
    flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=device)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
    return bool(int(flag.item()))


def flatten_grads(named_grads) -> torch.Tensor:
    return torch.cat([g.reshape(-1) for _, g in sorted(named_grads.items())])


class PeerGradExchange:
    """Symmetric (peer-mapped) gradient buffers for ``grapes_step_tail`` / ``grapes_allreduce_adam_peer``: every rank
    allocates the same buffer with ``torch.distributed._symmetric_memory`` and receives the peers' device pointers, so the
    mean all-reduce and both Adam updates run as ONE kernel over NVLink inside the step's CUDA graph (no host-side
    collective call).  ``embed_floats`` > 0 adds a second symmetric buffer of that many floats (``ebuf``, peers'
    pointers in ``embed_ptrs``): the payload of a learned node-feature table (``grapes_step_tail_embed``)."""

    def __init__(self, n_floats: int, device: torch.device, group=None, embed_floats: int = 0):
        import ctypes
        import torch.distributed._symmetric_memory as symm_mem
        from ._lib import lib
        group = group or dist.group.WORLD
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        if self.world > 8:
            raise RuntimeError("peer exchange is built for one NVSwitch box (<= 8 ranks)")
        total = int(lib().cdll.grapes_peer_buffer_floats(int(n_floats), self.world))
        self.buf = symm_mem.empty(total, dtype=torch.float32, device=device)
        self.buf.zero_()
        self.hdl = symm_mem.rendezvous(self.buf, group.group_name if hasattr(group, "group_name") else group)
        ptrs = [int(p) for p in self.hdl.buffer_ptrs]
        assert ptrs[self.rank] == self.buf.data_ptr()
        self.peer_ptrs = (ctypes.c_void_p * self.world)(*ptrs)              # HOST array handed to the C ABI
        self.ebuf, self.embed_ptrs = None, None
        if embed_floats > 0:
            self.ebuf = symm_mem.empty(int(embed_floats), dtype=torch.float32, device=device)
            self.ebuf.zero_()
            self.ehdl = symm_mem.rendezvous(self.ebuf, group.group_name if hasattr(group, "group_name") else group)
            eptrs = [int(p) for p in self.ehdl.buffer_ptrs]
            assert eptrs[self.rank] == self.ebuf.data_ptr()
            self.embed_ptrs = (ctypes.c_void_p * self.world)(*eptrs)
        self.state = torch.zeros(int(lib().cdll.grapes_peer_state_words()), dtype=torch.int32, device=device)
        torch.cuda.synchronize(device)
        # NOTE: no collective here.  The caller must synchronise the ranks once before the first exchange (every buffer is
        # zeroed before anyone publishes): GrapesEngine.enable_data_parallel does it with the all-reduce that also makes
        # the ranks agree on whether the peer mapping worked everywhere.


def eval_batches(num_batches: int, rank: int, world: int) -> List[int]:
    """Batches of the evaluation split that rank ``rank`` runs: every i with i mod W == rank, the tail round included
    (unlike :func:`shard_batches`, nothing waits on a per-batch collective here, so no batch is dropped)."""
    return list(range(rank, num_batches, world))


def allreduce_counts_(counts: torch.Tensor, group=None) -> torch.Tensor:
    """In-place integer sum over the ranks of ``group`` (hits / rows / tp / fp / fn): exact, so the scores computed from it
    are those of one process over all rows."""
    dist.all_reduce(counts, op=dist.ReduceOp.SUM, group=group)
    return counts


def gather_batch_predictions(local: torch.Tensor, batch_sizes: List[int], group=None) -> torch.Tensor:
    """The predictions of every batch in batch order, on every rank.  ``local`` holds this rank's batches
    (:func:`eval_batches`) back to back; ``batch_sizes`` lists the size of every batch of the split."""
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    per_rank = [sum(batch_sizes[i] for i in eval_batches(len(batch_sizes), r, world)) for r in range(world)]
    if local.numel() != per_rank[rank]:
        raise ValueError(f"rank {rank} holds {local.numel()} predictions, its batches have {per_rank[rank]}")
    width = max(per_rank + [1])
    padded = torch.zeros(width, dtype=local.dtype, device=local.device)
    padded[:local.numel()] = local
    parts = [torch.empty_like(padded) for _ in range(world)]
    dist.all_gather(parts, padded, group=group)
    out, cursor = [], [0] * world
    for i, n in enumerate(batch_sizes):
        r = i % world
        out.append(parts[r][cursor[r]:cursor[r] + n])
        cursor[r] += n
    return torch.cat(out) if out else local[:0]


class PeerRowTable:
    """A row table partitioned across the ranks of ``group`` -- the layer-2 operand of
    :func:`grapes_b200.gcn.full_graph_forward_sharded`, or a shard of the feature table (:class:`ShardedFeatures`): one
    ``torch.distributed._symmetric_memory`` buffer of ``rows`` x ``ld`` elements of ``dtype`` (fp32 or bf16) per rank (this
    rank's rows, zero pad columns), ``ptrs`` = the HOST array of every rank's buffer address (own at ``rank``), and ``barrier()`` = the
    stream-ordered barrier of the symmetric-memory handle (no host synchronisation).  Construction only allocates (rank
    local); :meth:`rendezvous` maps the peers and is collective.  Built once per graph and classifier width and cached
    with the window structure (``eval._sharded_eval``)."""

    def __init__(self, rows: int, ld: int, device: torch.device, group=None, dtype: torch.dtype = torch.float32):
        import torch.distributed._symmetric_memory as symm_mem
        self.group = group or dist.group.WORLD
        self.rank, self.world = dist.get_rank(self.group), dist.get_world_size(self.group)
        if self.world > 8:
            raise RuntimeError("the peer row table is built for one NVSwitch box (<= 8 ranks)")
        self.ld = int(ld)
        self.buf = symm_mem.empty(max(int(rows), 1) * self.ld, dtype=dtype, device=device)
        self.buf.zero_()
        self.rows = self.buf.view(max(int(rows), 1), self.ld)
        self.hdl, self.ptrs = None, None

    def rendezvous(self):
        import ctypes
        import torch.distributed._symmetric_memory as symm_mem
        g = self.group
        self.hdl = symm_mem.rendezvous(self.buf, g.group_name if hasattr(g, "group_name") else g)
        ptrs = [int(p) for p in self.hdl.buffer_ptrs]
        assert ptrs[self.rank] == self.buf.data_ptr()
        self.ptrs = (ctypes.c_void_p * self.world)(*ptrs)
        torch.cuda.synchronize(self.buf.device)
        return self

    def barrier(self):
        self.hdl.barrier(channel=0)


def feature_bounds(num_nodes: int, world: int) -> List[int]:
    """Row bounds of a feature table sharded between ``world`` ranks: equal contiguous ranges, bounds[r] = min(N, r *
    ceil(N / W)).  The table is sharded because it does not fit one device, so memory balance is the goal; the last
    ranges are short or empty when W does not divide N (N < W included)."""
    per = -(-int(num_nodes) // int(world))
    return [min(int(num_nodes), r * per) for r in range(int(world) + 1)]


def feature_pitch(num_features: int) -> int:
    """Row pitch (elements) of a feature shard: F rounded up to 4, the pitch the engine gives a replicated fp32 table;
    for bf16 it keeps every row 8-byte aligned.  The pad columns are zero."""
    return (int(num_features) + 3) // 4 * 4


def fill_plan(lo: int, hi: int, row_bytes: int, chunk_bytes: int = 1 << 30) -> List[Tuple[int, int]]:
    """Row ranges [a, b) covering [lo, hi) with at most ``chunk_bytes`` of source rows each (at least one row): the copies
    that fill one shard, so a host table is staged through at most that much device memory at a time."""
    step = max(1, int(chunk_bytes) // max(int(row_bytes), 1))
    return [(a, min(a + step, hi)) for a in range(int(lo), int(hi), step)]


class ShardedFeatures:
    """A feature table [N, F] sharded by rows across the data-parallel ranks (``train(..., shard_features=True)``): rank r
    holds rows ``bounds[r] .. bounds[r + 1]`` (:func:`feature_bounds`) in a :class:`PeerRowTable` of pitch ``ldx``
    (:func:`feature_pitch`, zero pad columns) and reads the other rows from their owners over NVLink peer memory.  Pass it
    as ``x`` to :class:`grapes_b200.engine.GrapesEngine` and as ``features`` to :func:`grapes_b200.eval.evaluate`; the
    results are bit-identical to those over the replicated table.

    Attributes: ``N``, ``F``, ``ldx``, ``dtype`` (fp32 or bf16, as ``x``), ``world``, ``rank``, ``bounds`` (W + 1 ints),
    ``table`` (``rows`` [max rows, ldx], ``ptrs`` = HOST array of every rank's shard), ``local`` = this rank's [rows, F]
    view, ``bounds_c`` = the bounds as a HOST int64 array for the C ABI.

    The constructor is collective over ``group`` (default: the world).  It fills this rank's rows from ``x[lo:hi]`` in
    chunks of at most ``chunk_bytes``; ``x`` may be a host tensor (memory-mapped or not) or a device tensor, and the whole
    table never goes to one device.  When the symmetric allocation or mapping fails on any rank, every rank raises
    ``GrapesError`` (agreed through :func:`ranks_agree`): there is no replicated fall-back, since the table may not fit.
    The shards are read-only once built; construction ends with a collective, so every shard is filled before any rank
    reads a peer's."""

    def __init__(self, x: torch.Tensor, device, group=None, chunk_bytes: int = 1 << 30):
        from ._lib import GrapesError
        device = torch.device(device)
        self.group = group or dist.group.WORLD
        world, rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        self._shape(x, world, rank)
        rows = max(self.bounds[r + 1] - self.bounds[r] for r in range(world))
        table, why = None, ""
        try:
            table = PeerRowTable(rows, self.ldx, device, self.group, dtype=self.dtype)
        except Exception as exc:                        # noqa: BLE001 -- agreed below and raised on every rank
            why = f"{type(exc).__name__}: {exc}"
        if ranks_agree(table is not None, device, self.group):
            try:
                table.rendezvous()
            except Exception as exc:                    # noqa: BLE001
                why, table = f"{type(exc).__name__}: {exc}", None
            if not ranks_agree(table is not None, device, self.group):
                table = None
        else:
            table = None
        if table is None:
            raise GrapesError("sharded feature table: symmetric allocation or peer mapping failed " +
                              (f"on this rank ({why})" if why else "on another rank"))
        self.table = table
        self._fill(x, chunk_bytes)
        torch.cuda.synchronize(device)
        ranks_agree(True, device, self.group)           # every shard is filled before any rank reads a peer's

    def _shape(self, x, world: int, rank: int):
        from ._lib import GrapesError
        if x.dim() != 2 or x.dtype not in (torch.float32, torch.bfloat16):
            raise GrapesError("a sharded feature table is a 2-D fp32 or bf16 tensor")
        if not 1 <= world <= 8:
            raise GrapesError(f"a sharded feature table spans 1 to 8 ranks (one NVSwitch box), not {world}")
        self.N, self.F = int(x.shape[0]), int(x.shape[1])
        self.dtype, self.world, self.rank = x.dtype, int(world), int(rank)
        self.ldx = feature_pitch(self.F)
        self.bounds = feature_bounds(self.N, world)
        self.lo, self.hi = self.bounds[rank], self.bounds[rank + 1]

    def _fill(self, x: torch.Tensor, chunk_bytes: int):
        import ctypes
        self.local = self.table.rows[:self.hi - self.lo, :self.F]
        for a, b in fill_plan(self.lo, self.hi, self.F * x.element_size(), chunk_bytes):
            self.local[a - self.lo:b - self.lo].copy_(x[a:b])
        self.bounds_c = (ctypes.c_int64 * (self.world + 1))(*self.bounds)

    @property
    def ptrs(self):
        return self.table.ptrs

    @property
    def x_bf16(self) -> bool:
        return self.dtype == torch.bfloat16

    @property
    def table_bytes(self) -> int:
        """Device bytes of this rank's shard (pad columns included)."""
        return self.table.rows.numel() * self.table.rows.element_size()

    @classmethod
    def emulate(cls, x: torch.Tensor, world: int, device=None, chunk_bytes: int = 1 << 30) -> List["ShardedFeatures"]:
        """One-process stand-in: the W shards in W allocations of one device (:class:`grapes_b200.gcn.LocalRowTable`), one
        holder per emulated rank, all sharing them; any one of them serves an engine, which then reads all W."""
        from .gcn import LocalRowTable
        device = torch.device(device) if device is not None else x.device
        out = []
        for r in range(int(world)):
            s = cls.__new__(cls)
            s.group = None
            s._shape(x, int(world), r)
            out.append(s)
        rows = max(out[0].bounds[r + 1] - out[0].bounds[r] for r in range(int(world)))
        tables = LocalRowTable.make(int(world), rows, out[0].ldx, device, dtype=x.dtype)
        for s, t in zip(out, tables):
            s.table = t
            s._fill(x, chunk_bytes)
        return out


class ShardedEmbedding(ShardedFeatures):
    """A LEARNED node-feature table [N, F] (``--embed_nodes``; fp32, F % 4 == 0) sharded by rows across the data-parallel
    ranks (``train(..., shard_embeddings=True)``): rank r holds rows ``bounds[r] .. bounds[r + 1]`` as
    :class:`ShardedFeatures` does, plus the two Adam moments of those rows (``exp_avg``, ``exp_avg_sq``: [rows, F], zero at
    the start, ordinary device memory) and updates only those rows (``grapes_embed_merge_adam_rows``).  Every step posts
    a table epoch into a small symmetric buffer (``epoch``; ``epoch_ptrs`` = the HOST array of every rank's), and every
    read of the table waits for every peer's post of the previous step (``grapes_embed_epoch_post`` / ``_wait``; the
    ordering argument is in csrc/peer_comm.cu).  Results are bit-identical to the replicated learned table.

    The constructor is collective, with :class:`ShardedFeatures`' fill and its rule of agreeing on failure (every rank
    raises ``GrapesError`` when any rank cannot allocate or map).  :meth:`to_dense` returns the [N, F] table (collective
    under a group).  :meth:`emulate` is the one-process stand-in: W shards with their moments on one device, no epoch."""

    def __init__(self, x: torch.Tensor, device, group=None, chunk_bytes: int = 1 << 30):
        import ctypes
        from ._lib import GrapesError, lib
        self._check(x)
        super().__init__(x, device, group, chunk_bytes)
        device = torch.device(device)
        self._moments(device)
        self.shards = None
        buf, why = None, ""
        try:
            import torch.distributed._symmetric_memory as symm_mem
            buf = symm_mem.empty(int(lib().cdll.grapes_embed_epoch_words(self.world)), dtype=torch.int32, device=device)
            buf.zero_()
            hdl = symm_mem.rendezvous(buf, self.group.group_name if hasattr(self.group, "group_name") else self.group)
            ptrs = [int(p) for p in hdl.buffer_ptrs]
            assert ptrs[self.rank] == buf.data_ptr()
        except Exception as exc:                        # noqa: BLE001 -- agreed below and raised on every rank
            why, buf = f"{type(exc).__name__}: {exc}", None
        torch.cuda.synchronize(device)
        if not ranks_agree(buf is not None, device, self.group):   # also: every epoch buffer is zero before any post
            raise GrapesError("sharded learned table: symmetric epoch buffer could not be mapped " +
                              (f"on this rank ({why})" if why else "on another rank"))
        self.epoch, self._epoch_hdl = buf, hdl
        self.epoch_ptrs = (ctypes.c_void_p * self.world)(*ptrs)

    @staticmethod
    def _check(x):
        from ._lib import GrapesError
        if x.dim() != 2 or x.dtype != torch.float32 or int(x.shape[1]) % 4 != 0:
            raise GrapesError("a sharded learned table is a 2-D fp32 tensor whose width is a multiple of 4")

    def _moments(self, device):
        rows = max(self.hi - self.lo, 1)
        self.exp_avg = torch.zeros((rows, self.F), dtype=torch.float32, device=device)
        self.exp_avg_sq = torch.zeros((rows, self.F), dtype=torch.float32, device=device)

    def load_rows(self, x: torch.Tensor, exp_avg: torch.Tensor, exp_avg_sq: torch.Tensor, chunk_bytes: int = 1 << 30):
        """Overwrites this rank's rows of the table and of both moments in place from [N, F] sources (host,
        memory-mapped or device; a checkpoint's ``table_source``), in chunks of at most ``chunk_bytes``."""
        n = self.hi - self.lo
        for a, b in fill_plan(self.lo, self.hi, self.F * 4, chunk_bytes):
            for dst, src in ((self.table.rows[:n, :self.F], x), (self.exp_avg, exp_avg), (self.exp_avg_sq, exp_avg_sq)):
                dst[a - self.lo:b - self.lo].copy_(src[a:b])

    @property
    def moment_bytes(self) -> int:
        """Device bytes of this rank's two moment arrays."""
        return 2 * self.exp_avg.numel() * self.exp_avg.element_size()

    @classmethod
    def emulate(cls, x: torch.Tensor, world: int, device=None, chunk_bytes: int = 1 << 30) -> List["ShardedEmbedding"]:
        cls._check(x)
        out = super().emulate(x, world, device, chunk_bytes)
        for s in out:
            s._moments(s.table.rows.device)
            s.shards, s.epoch, s.epoch_ptrs = out, None, None
        return out

    def _dense(self, local_of) -> torch.Tensor:
        """[N, F] from every rank's [rows, F] array ``local_of(holder)`` (all-gather under a group)."""
        if self.shards is not None:
            return torch.cat([local_of(s)[:s.hi - s.lo] for s in self.shards])
        rows = max(self.bounds[r + 1] - self.bounds[r] for r in range(self.world))
        mine = torch.zeros((max(rows, 1), self.F), dtype=torch.float32, device=self.exp_avg.device)
        mine[:self.hi - self.lo].copy_(local_of(self)[:self.hi - self.lo])
        parts = [torch.empty_like(mine) for _ in range(self.world)]
        dist.all_gather(parts, mine, group=self.group)
        return torch.cat([parts[r][:self.bounds[r + 1] - self.bounds[r]] for r in range(self.world)])

    def to_dense(self) -> torch.Tensor:
        """The whole [N, F] table (a new tensor on this device); collective under a group."""
        return self._dense(lambda s: s.table.rows[:, :s.F])

    def moments_dense(self) -> Tuple[torch.Tensor, torch.Tensor]:
        """Both Adam moments of the whole table, [N, F] each; collective under a group."""
        return self._dense(lambda s: s.exp_avg), self._dense(lambda s: s.exp_avg_sq)
