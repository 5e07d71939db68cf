"""Checkpoint and resume of a training run: the parameters, both Adam optimisers, the device Philox counters of the sampler
and of dropout, the learned node-feature table with its moments (``--embed_nodes``, replicated or sharded across the
ranks) and the loop position of ``train()``.  A run interrupted and resumed from a checkpoint computes the same bits
as one that never stopped.

A checkpoint is a directory ``<checkpoint_dir>/step-<global step, 9 digits>/``:

  ``meta.json``      rank 0, written last: format, world size, exchange, sharding flags, the ``Arguments``, the shapes
                     (N, F, C, D, H, k, B, feature dtype, embed_nodes, multilabel, n_par), the loop position (epoch,
                     batches done in it, global step), the byte size of every other file and a CRC32 of every small one
  ``model.pt``       rank 0: ``{"gcn_c", "gcn_gf", "gcn_z"}``, PyG-named state dicts on the CPU; they load into
                     ``grapes_b200.gcn.GCN`` and into the reference's ``GCN``
  ``optim.pt``       rank 0: the flat ``exp_avg``, ``exp_avg_sq`` (length n_par) and ``adam_steps`` [2]
  ``rank<r>.pt``     every rank: ``rng_state``, ``drop_state`` and the loop state (``acc_c``, ``acc_gfn``, the last step log)
  ``table.f32``, ``table_m.f32``, ``table_v.f32``
                     ``--embed_nodes`` only: the table and its two Adam moments as raw little-endian float32 [N, F],
                     row-major, no header.  Each owner writes its own rows at their offsets (a sharded table: every rank
                     its shard; a replicated one: rank 0 all rows), so nothing is gathered onto one device or host, and
                     any world size reads any rows back through ``np.memmap`` (:func:`table_source`).

Atomicity: every rank writes into ``step-….tmp/`` and fsyncs its files; after a barrier rank 0 writes ``meta.json``,
fsyncs it and the directory, renames ``….tmp`` to ``step-…`` and replaces ``LATEST`` (a temporary file, then
``os.replace``); then the two newest checkpoints are kept and older ones deleted.  A crash at any point leaves
``LATEST`` naming a complete checkpoint.

The engine's captured CUDA graphs hold raw pointers to every tensor a checkpoint restores, so :func:`load` copies into
the existing tensors and never rebinds one: a graph captured before the load replays the loaded state."""
from __future__ import annotations

import json
import os
import re
import shutil
import warnings
import zlib
from typing import Dict, Optional, Tuple

import numpy as np
import torch
import torch.distributed as dist

from ._lib import GrapesError
from .dist import fill_plan, ranks_agree

FORMAT = 1
TABLE_FILES = ("table.f32", "table_m.f32", "table_v.f32")
#: meta fields that must equal the loading engine's
SHAPE_FIELDS = ("N", "F", "C", "D", "H", "k", "B", "dtype", "embed_nodes", "multilabel", "n_par")
#: meta fields that may differ, with a warning: the trajectory of the resumed run differs from the saved run's (batch
#: sharding depends on the world size; the peer and NCCL means round differently)
LAYOUT_FIELDS = ("world", "exchange", "shard_features", "shard_embeddings")
#: ``Arguments`` fields that may differ between the saved run and the resumed one; every other field must match
FREE_ARGS = ("max_epochs", "eval_frequency", "runs", "notes", "log_wandb", "config_file")
_STEP_RE = re.compile(r"^step-(\d{9})$")


def step_path(checkpoint_dir: str, step: int) -> str:
    return os.path.join(checkpoint_dir, f"step-{int(step):09d}")


def _fsync_path(path: str):
    fd = os.open(path, os.O_RDONLY)
    try:
        os.fsync(fd)
    finally:
        os.close(fd)


def _crc(path: str) -> int:
    c = 0
    with open(path, "rb") as f:
        for blk in iter(lambda: f.read(1 << 24), b""):
            c = zlib.crc32(blk, c)
    return c


def _torch_save(obj, path: str):
    with open(path, "wb") as f:
        torch.save(obj, f)
        f.flush()
        os.fsync(f.fileno())


def _complete(path: str) -> bool:
    return os.path.isfile(os.path.join(path, "meta.json"))


def latest(checkpoint_dir: str) -> Optional[str]:
    """The checkpoint ``LATEST`` names, or None when there is none.  When ``LATEST`` names a directory that is gone (a
    checkpoint of the same step being replaced when the process died), the newest complete ``step-…`` directory."""
    try:
        with open(os.path.join(checkpoint_dir, "LATEST")) as f:
            name = f.read().strip()
    except FileNotFoundError:
        name = None
    if name and _STEP_RE.match(name) and _complete(os.path.join(checkpoint_dir, name)):
        return os.path.join(checkpoint_dir, name)
    try:
        names = sorted(n for n in os.listdir(checkpoint_dir) if _STEP_RE.match(n))
    except FileNotFoundError:
        return None
    done = [n for n in names if _complete(os.path.join(checkpoint_dir, n))]
    return os.path.join(checkpoint_dir, done[-1]) if done else None


def _resolve(path: str) -> str:
    """A checkpoint directory as given, or the latest checkpoint of a checkpoint root."""
    if _complete(path):
        return path
    found = latest(path)
    if found is None:
        raise GrapesError(f"no complete checkpoint at {path}")
    return found


def read_meta(path: str) -> dict:
    with open(os.path.join(_resolve(path), "meta.json")) as f:
        return json.load(f)


def read_rows(path: str, num_rows: int, num_cols: int) -> torch.Tensor:
    """A raw little-endian float32 [num_rows, num_cols] file as a read-only memory-mapped CPU tensor."""
    want = 4 * int(num_rows) * int(num_cols)
    have = os.path.getsize(path)
    if have != want:
        raise GrapesError(f"{os.path.basename(path)}: {have} bytes, a [{num_rows}, {num_cols}] float32 table has {want}")
    if want == 0:
        return torch.zeros((int(num_rows), int(num_cols)), dtype=torch.float32)
    arr = np.memmap(path, dtype="<f4", mode="r", shape=(int(num_rows), int(num_cols)))
    with warnings.catch_warnings():                 # read-only mapping: every consumer only copies from it
        warnings.simplefilter("ignore", UserWarning)
        return torch.from_numpy(arr)


def table_source(path: str) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """The learned table of a checkpoint and its two Adam moments, each a memory-mapped [N, F] CPU tensor: any rank of
    any world size reads its rows from them (``ShardedFeatures`` fills a shard from such a tensor)."""
    path = _resolve(path)
    meta = read_meta(path)
    if not meta["embed_nodes"]:
        raise GrapesError(f"checkpoint {path} holds no learned node-feature table (saved without embed_nodes)")
    return tuple(read_rows(os.path.join(path, n), meta["N"], meta["F"]) for n in TABLE_FILES)


def write_rows(path: str, rows: torch.Tensor, row0: int, num_rows: int, chunk_bytes: int = 1 << 30):
    """Writes ``rows`` ([n, F] float32, host or device) as rows ``[row0, row0 + n)`` of the raw [num_rows, F] file at
    ``path`` (created at its full size when missing), with ``pwrite`` in chunks of at most ``chunk_bytes``
    (:func:`grapes_b200.dist.fill_plan`); device rows go through one pinned staging buffer.  Several owners may write
    disjoint rows of one file concurrently.  The file is fsynced."""
    n, F = int(rows.shape[0]), int(rows.shape[1])
    row_bytes = 4 * F
    if rows.dtype != torch.float32 or not 0 <= row0 <= row0 + n <= num_rows:
        raise GrapesError(f"rows [{row0}, {row0 + n}) of float32 [{num_rows}, {F}]: got {rows.dtype}")
    fd = os.open(path, os.O_WRONLY | os.O_CREAT, 0o644)
    try:
        if os.fstat(fd).st_size < num_rows * row_bytes:
            os.ftruncate(fd, num_rows * row_bytes)     # never shrinks: every owner extends it to the same size
        staging = None
        for a, b in fill_plan(row0, row0 + n, row_bytes, chunk_bytes):
            src = rows[a - row0:b - row0]
            if src.is_cuda:
                if staging is None:
                    per = max(1, int(chunk_bytes) // row_bytes)
                    staging = torch.empty(min(per, n) * F, dtype=torch.float32, pin_memory=True)
                buf = staging[:(b - a) * F].view(b - a, F)
                buf.copy_(src)                         # synchronous: the device rows are in host memory afterwards
                arr = buf.numpy()
            else:
                arr = src.contiguous().numpy()
            mv = memoryview(np.ascontiguousarray(arr, dtype="<f4").reshape(-1).view(np.uint8))
            off = a * row_bytes
            while len(mv):
                k = os.pwrite(fd, mv, off)
                mv, off = mv[k:], off + k
        os.fsync(fd)
    finally:
        os.close(fd)


# ---------------------------------------------------------------------------------------------------- meta
def _group(engine, group):
    if group is not None:
        return group
    if engine.dp_world > 1:
        return engine.dp_group or dist.group.WORLD
    return None


def _agree(ok: bool, device, group) -> bool:
    if group is None:
        return ok
    if dist.get_backend(group) == "gloo":
        device = torch.device("cpu")
    return ranks_agree(ok, device, group)


def describe(engine) -> dict:
    """The fields of ``meta.json`` that describe the engine: its shapes and its data-parallel layout."""
    es = engine.embed_shards
    return dict(N=int(engine.N), F=int(engine.F), C=int(engine.C), D=int(engine.D), H=int(engine.H), k=int(engine.k),
                B=int(engine.B), dtype="bfloat16" if engine.x_bf16 else "float32", embed_nodes=bool(engine.embed_nodes),
                multilabel=bool(engine.multilabel), n_par=int(engine.n_par), world=int(engine.dp_world),
                exchange="peer" if engine.peer is not None else ("nccl" if engine.dp_group is not None else None),
                shard_features=engine.features is not None and es is None, shard_embeddings=es is not None)


def _args_dict(args) -> Optional[dict]:
    if args is None:
        return None
    return dict(args.as_dict() if hasattr(args, "as_dict") else args)


def check_meta(meta: dict, current: dict, args=None):
    """Refuses (``GrapesError`` naming the field) a checkpoint whose format, shapes or ``Arguments`` (except
    :data:`FREE_ARGS`) differ from ``current`` (:func:`describe` of the loading engine) and ``args``; warns when the world
    size, the exchange or a sharding flag differs.  ``args`` None: the ``Arguments`` are not compared."""
    if meta.get("format") != FORMAT:
        raise GrapesError(f"checkpoint format: {meta.get('format')!r}, this build reads {FORMAT}")
    for key in SHAPE_FIELDS:
        if meta.get(key) != current[key]:
            raise GrapesError(f"checkpoint {key} = {meta.get(key)!r}, the engine has {current[key]!r}")
    a = _args_dict(args)
    saved = meta.get("args")
    if a is not None and saved is not None:
        for key in sorted(set(a) | set(saved)):
            if key not in FREE_ARGS and a.get(key) != saved.get(key):
                raise GrapesError(f"checkpoint was saved with {key} = {saved.get(key)!r}, this run has {a.get(key)!r}")
    changed = [f"{k} {meta.get(k)!r} -> {current[k]!r}" for k in LAYOUT_FIELDS if meta.get(k) != current[k]]
    if changed:
        warnings.warn("grapes_b200: resuming with " + ", ".join(changed) + ": the trajectory will differ from that of "
                      "the saved run")


def check_files(path: str, meta: dict):
    """Refuses a checkpoint whose files do not have the sizes ``meta.json`` records, or whose small files fail their
    CRC32."""
    for name, size in meta["sizes"].items():
        p = os.path.join(path, name)
        if not os.path.isfile(p) or os.path.getsize(p) != size:
            have = os.path.getsize(p) if os.path.isfile(p) else None
            raise GrapesError(f"checkpoint file {name}: {have} bytes, meta.json records {size}")
    for name, crc in meta["crc"].items():
        if _crc(os.path.join(path, name)) != crc:
            raise GrapesError(f"checkpoint file {name}: CRC32 mismatch")


# ---------------------------------------------------------------------------------------------------- save / load
def _holders(engine):
    es = engine.embed_shards
    return es.shards if es.shards is not None else [es]


def save(engine, checkpoint_dir: str, loop_state: Optional[dict] = None, *, args=None, group=None) -> str:
    """Writes a checkpoint of ``engine`` as ``<checkpoint_dir>/step-<step>/`` and points ``LATEST`` at it; returns its
    path.  Collective over the engine's data-parallel group (``group`` overrides it).

    ``loop_state`` (optional): ``epoch``, ``batch`` (batches of that epoch done), ``step`` (global step; default: the
    optimiser step count), ``acc_c``, ``acc_gfn``, ``last`` (the last step log) -- what ``train()`` resumes from.
    ``args``: the run's ``Arguments``, recorded so that a resume can refuse a different configuration.

    It synchronises the device first and refuses (``GrapesError`` on every rank) when a step's flag word is non-zero
    (overflow, failed or sticky exchange), when the ranks' parameters differ (int64 checksum of the parameter bits), or
    when the target directory exists and is not a checkpoint."""
    group = _group(engine, group)
    rank = dist.get_rank(group) if group is not None else 0
    dev = engine.device
    if dev.type == "cuda":
        torch.cuda.synchronize(dev)
    loop = dict(loop_state or {})
    step = int(loop.get("step", int(engine.adam_steps[0].item())))
    loop.setdefault("step", step)
    final = step_path(checkpoint_dir, step)
    tmp = final + ".tmp"

    why = None
    flags = int(engine.overflow.item()) | int(engine.scal[15].item())
    if flags:
        why = f"a step's flag word is {flags:#x} (overflow or failed exchange): the state is not a training state"
    elif os.path.exists(final) and not _complete(final):
        why = f"{final} exists and is not a checkpoint"
    if not _agree(why is None, dev, group):
        raise GrapesError("checkpoint refused: " + (why or "refused on another rank"))
    if group is not None:
        s = engine.params.view(torch.int32).to(torch.int64).sum().reshape(1)
        if dist.get_backend(group) == "gloo":
            s = s.cpu()
        lo, hi = s.clone(), s.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN, group=group)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX, group=group)
        if int(lo.item()) != int(hi.item()):
            raise GrapesError("checkpoint refused: the ranks' parameters differ (checksums "
                              f"{int(lo.item())} .. {int(hi.item())})")

    err = None
    if rank == 0:
        try:
            os.makedirs(checkpoint_dir, exist_ok=True)
            shutil.rmtree(tmp, ignore_errors=True)     # left by a save that died
            os.mkdir(tmp)
        except OSError as exc:
            err = exc
    if not _agree(err is None, dev, group):
        raise GrapesError(f"checkpoint: cannot create {tmp}" + (f" ({err})" if err else " (on rank 0)"))

    try:
        if rank == 0:
            _torch_save({k: {n: t.detach().cpu().clone() for n, t in v.items()}
                         for k, v in engine.state_dicts().items()}, os.path.join(tmp, "model.pt"))
            _torch_save({"exp_avg": engine.exp_avg.cpu(), "exp_avg_sq": engine.exp_avg_sq.cpu(),
                         "adam_steps": engine.adam_steps.cpu()}, os.path.join(tmp, "optim.pt"))
        _torch_save({"rng_state": engine.rng_state.cpu(), "drop_state": engine.drop_state.cpu(),
                     "loop": {k: loop.get(k) for k in ("acc_c", "acc_gfn", "last")}},
                    os.path.join(tmp, f"rank{rank}.pt"))
        if engine.embed_nodes:
            N, F = engine.N, engine.F
            paths = [os.path.join(tmp, n) for n in TABLE_FILES]
            if engine.embed_shards is not None:
                for s in _holders(engine):
                    n = s.hi - s.lo
                    for p, t in zip(paths, (s.table.rows[:n, :F], s.exp_avg[:n], s.exp_avg_sq[:n])):
                        write_rows(p, t, s.lo, N)
            elif rank == 0:
                for p, t in zip(paths, (engine.x, engine.emb_exp_avg, engine.emb_exp_avg_sq)):
                    write_rows(p, t, 0, N)
    except OSError as exc:
        err = exc
    if not _agree(err is None, dev, group):               # every rank's files are written and fsynced
        raise GrapesError("checkpoint: writing failed " + (f"on this rank ({err})" if err else "on another rank"))

    if rank == 0:
        try:
            _commit(engine, checkpoint_dir, tmp, final, loop, args, group)
        except OSError as exc:
            err = exc
    if not _agree(err is None, dev, group):               # nobody returns before the checkpoint exists
        raise GrapesError("checkpoint: committing failed " + (f"({err})" if err else "on rank 0"))
    return final


def _commit(engine, checkpoint_dir, tmp, final, loop, args, group):
    """Rank 0, after every rank's files are durable: meta.json, the rename, LATEST, and the deletion of old
    checkpoints."""
    names = sorted(os.listdir(tmp))
    meta = dict(format=FORMAT, **describe(engine), args=_args_dict(args),
                epoch=loop.get("epoch"), batch=loop.get("batch"), step=int(loop["step"]),
                sizes={n: os.path.getsize(os.path.join(tmp, n)) for n in names},
                crc={n: _crc(os.path.join(tmp, n)) for n in names if n not in TABLE_FILES})
    if group is not None:
        meta["world"] = dist.get_world_size(group)
    with open(os.path.join(tmp, "meta.json"), "w") as f:
        json.dump(meta, f, indent=1, sort_keys=True)
        f.flush()
        os.fsync(f.fileno())
    _fsync_path(tmp)
    prev = latest(checkpoint_dir)
    old = None
    if os.path.exists(final):                             # the same step saved again: the new one replaces it
        old = final + ".old"
        shutil.rmtree(old, ignore_errors=True)
        os.rename(final, old)
    os.rename(tmp, final)
    _fsync_path(checkpoint_dir)
    lt = os.path.join(checkpoint_dir, "LATEST.tmp")
    with open(lt, "w") as f:
        f.write(os.path.basename(final) + "\n")
        f.flush()
        os.fsync(f.fileno())
    os.replace(lt, os.path.join(checkpoint_dir, "LATEST"))
    _fsync_path(checkpoint_dir)
    keep = {os.path.basename(final)} | ({os.path.basename(prev)} if prev else set())
    for n in os.listdir(checkpoint_dir):
        if (_STEP_RE.match(n) and n not in keep) or (old is not None and n == os.path.basename(old)):
            shutil.rmtree(os.path.join(checkpoint_dir, n), ignore_errors=True)


def load(engine, path: str, *, args=None, group=None) -> dict:
    """Restores a checkpoint into ``engine`` in place and returns its loop state (``epoch``, ``batch``, ``step``,
    ``acc_c``, ``acc_gfn``, ``last``).  ``path``: a checkpoint, or a checkpoint directory (its latest checkpoint).
    Collective over the engine's data-parallel group (``group`` overrides it).

    Every restored tensor is overwritten with ``copy_`` (captured graphs keep their pointers); a prefetched front end is
    dropped; the exchange state (peer slots, parity, state words, the table epoch) is not touched.  ``meta.json`` is
    checked against the engine and ``args`` (:func:`check_meta`) and the files against their sizes and CRCs
    (:func:`check_files`); any mismatch raises ``GrapesError`` on every rank.  A learned table is read through
    :func:`table_source`: every rank copies only its own rows, whatever world size saved it."""
    group = _group(engine, group)
    rank = dist.get_rank(group) if group is not None else 0
    dev = engine.device
    err, meta = None, None
    try:
        path = _resolve(path)
        meta = read_meta(path)
        check_meta(meta, describe(engine) | ({"world": dist.get_world_size(group)} if group is not None else {}), args)
        check_files(path, meta)
    except (GrapesError, OSError, ValueError, KeyError) as exc:
        err = exc
    if not _agree(err is None, dev, group):
        raise GrapesError(f"checkpoint {path} refused: " + (str(err) if err is not None else "refused on another rank"))

    if dev.type == "cuda":
        torch.cuda.synchronize(dev)
    model = torch.load(os.path.join(path, "model.pt"), map_location="cpu", weights_only=True)
    engine.load_state_dicts(**model)
    optim = torch.load(os.path.join(path, "optim.pt"), map_location="cpu", weights_only=True)
    for name in ("exp_avg", "exp_avg_sq", "adam_steps"):
        getattr(engine, name).copy_(optim[name])
    src = rank if rank < int(meta["world"]) else 0       # another world size: rank 0's counters (every rank's are equal)
    rs = torch.load(os.path.join(path, f"rank{src}.pt"), map_location="cpu", weights_only=True)
    engine.rng_state.copy_(rs["rng_state"])
    engine.drop_state.copy_(rs["drop_state"])
    if engine.embed_nodes:
        table, m, v = table_source(path)
        if engine.embed_shards is not None:
            for s in _holders(engine):
                s.load_rows(table, m, v)
        else:
            for dst, t in ((engine.x, table), (engine.emb_exp_avg, m), (engine.emb_exp_avg_sq, v)):
                for a, b in fill_plan(0, engine.N, 4 * engine.F):
                    dst[a:b].copy_(t[a:b])
    engine._front_ready = [False, False]
    engine._pref_key = None
    if dev.type == "cuda":
        torch.cuda.synchronize(dev)
    _agree(True, dev, group)
    out = dict(rs["loop"])
    out.update(epoch=meta["epoch"], batch=meta["batch"], step=meta["step"])
    return out
