"""Dropout of the classifier GCN (modules/gcn.py:33,37) as the device engine draws it, restated in numpy, and the replay of
given masks inside the CPU oracle.

The keep bit of entry i = row * width + col of a site is Philox4x32-10 (Salmon et al. 2011) with counter
(i // 4, tag, step_lo, step_hi) and key (seed_lo, seed_hi), word i % 4; the entry is kept iff the word's 24 low bits are
below threshold = llrint((1 - p) * 2**24).  tag = 1 + site + 2 * rank, site 0 = hidden layer, 1 = logits.

The oracle (oracle/reference_port.py) applies dropout through its module-level ``F_.dropout``.  :func:`replay_masks`
swaps that name for the duration of a block: every call with p > 0 in training mode returns ``x * (keep / (1 - p))`` --
exactly what torch's CPU dropout computes from its Bernoulli draw ``keep`` -- with ``keep`` supplied by the caller; every
other call goes to torch unchanged."""
import contextlib

import numpy as np
import torch

from oracle import reference_port as rp

_M0, _M1, _W0, _W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
_U32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """ctr: 4 arrays (or ints) of uint32 values, key: 2 ints -> the 4 output words as uint64 arrays."""
    x0, x1, x2, x3 = np.broadcast_arrays(*(np.asarray(c, dtype=np.uint64) for c in ctr))
    k0, k1 = np.uint64(key[0]), np.uint64(key[1])
    for _ in range(10):
        p0 = np.uint64(_M0) * x0                        # < 2**64: exact in uint64
        p1 = np.uint64(_M1) * x2
        x0, x1, x2, x3 = (p1 >> np.uint64(32)) ^ x1 ^ k0, p1 & _U32, (p0 >> np.uint64(32)) ^ x3 ^ k1, p0 & _U32
        k0, k1 = (k0 + np.uint64(_W0)) & _U32, (k1 + np.uint64(_W1)) & _U32
    return x0, x1, x2, x3


def threshold(p: float) -> int:
    """llrint((1 - p) * 2**24): round half to even, like the engine's host code"""
    return int(np.rint((1.0 - p) * (1 << 24)))


def tag(site: int, rank: int = 0) -> int:
    return 1 + site + 2 * rank


def keep_mask(seed: int, step: int, site_tag: int, thr: int, rows: int, width: int) -> np.ndarray:
    """bool [rows, width]: the keep bits of one dropout site"""
    n = rows * width
    g = np.arange((n + 3) // 4, dtype=np.uint64)
    words = philox4x32_10((g, site_tag, step & 0xFFFFFFFF, step >> 32), (seed & 0xFFFFFFFF, seed >> 32))
    w = np.stack(words, axis=1).reshape(-1)[:n]
    return ((w & np.uint64(0xFFFFFF)) < np.uint64(thr)).reshape(rows, width)


def engine_masks(seed: int, step: int, p: float, rank: int = 0):
    """masks_for(site, shape) of the engine's step `step` (for :func:`replay_masks`)"""
    return lambda site, shape: torch.from_numpy(keep_mask(seed, step, tag(site, rank), threshold(p), *shape))


@contextlib.contextmanager
def replay_masks(masks_for):
    """Inside the block the oracle's dropout calls (p > 0, training) use ``masks_for(site, shape)`` (bool) as their
    Bernoulli draw; site alternates 0 (hidden layer), 1 (logits), as gcn_c's forward calls them."""
    real = rp.F_
    calls = [0]

    class _Dropout:
        def __getattr__(self, name):
            return getattr(real, name)

        @staticmethod
        def dropout(x, p=0.5, training=True, inplace=False):
            if not training or p == 0:
                return real.dropout(x, p=p, training=training, inplace=inplace)
            site = calls[0] % 2
            calls[0] += 1
            if p == 1:
                return x * torch.zeros((), dtype=x.dtype)          # torch: input * 0
            keep = masks_for(site, tuple(x.shape)).to(x.dtype)
            return x * (keep / (1 - p))

    rp.F_ = _Dropout()
    try:
        yield
    finally:
        rp.F_ = real
