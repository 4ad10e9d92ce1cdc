"""Host-side reference of the attention-dropout mask: a NumPy transcription of csrc/dropout_rng.cuh.

Every kernel regenerates the mask from (seed, offset, item, query i, key j) without storing it.  One Philox4x32-10 call
covers the 2 x 2 block (i >> 1, j >> 1) of an item:
    counter = (j >> 1, i >> 1, item, offset & 0xffffffff),   key = (seed_lo, seed_hi ^ offset_hi)
and word (i & 1) * 2 + (j & 1) of its output decides element (i, j): kept iff (word >> 8) >= ceil(float32(p) * 2^24).
A kept probability is scaled by float32(1 / (1 - p)).

Items: multi-head attention b * nH + h; window attention (b * nW + w) * nH + h, windows w counted row-major in the
shifted frame and i, j the row-major positions in the window (the order of window_partition_nd(cyclic_shift_nd(x))).

Vectorised over arrays of counters: products of two 32-bit words are formed in uint64 and cannot overflow.
"""
from __future__ import annotations

import math

import numpy as np

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
_LO = np.uint64(0xFFFFFFFF)
_S32 = np.uint64(32)


def philox4x32_10(ctr, key) -> np.ndarray:
    """ctr (..., 4) and key (..., 2) of 32-bit words (broadcast against each other) -> (..., 4) uint32."""
    ctr = np.asarray(ctr, dtype=np.uint64)
    key = np.asarray(key, dtype=np.uint64)
    c0, c1, c2, c3 = (ctr[..., n] for n in range(4))
    k0, k1 = key[..., 0], key[..., 1]
    for _ in range(10):
        p0, p1 = _M0 * c0, _M1 * c2
        c0, c1, c2, c3 = (p1 >> _S32) ^ c1 ^ k0, p1 & _LO, (p0 >> _S32) ^ c3 ^ k1, p0 & _LO
        k0, k1 = (k0 + _W0) & _LO, (k1 + _W1) & _LO
    return np.stack(np.broadcast_arrays(c0, c1, c2, c3), axis=-1).astype(np.uint32)


def dropout_threshold(p: float) -> int:
    """ceil(float32(p) * 2^24) in float32 arithmetic, as make_dropout computes it; 0 for p <= 0."""
    if p <= 0.0:
        return 0
    return math.ceil(float(np.float32(p) * np.float32(16777216.0)))


def keep_scale(p: float, seed: int, offset: int, item, i, j) -> np.ndarray:
    """0 or float32(1 / (1 - p)) for every (item, i, j) of the broadcast integer arrays item, i, j (float32)."""
    item, i, j = (np.asarray(x, dtype=np.uint64) for x in (item, i, j))
    inv_keep = np.float32(1.0) / (np.float32(1.0) - np.float32(p))
    if p <= 0.0:
        return np.broadcast_to(np.float32(1.0), np.broadcast_shapes(item.shape, i.shape, j.shape)).copy()
    seed, offset = int(seed) & 0xFFFFFFFFFFFFFFFF, int(offset) & 0xFFFFFFFFFFFFFFFF
    one = np.uint64(1)
    item, i, j = np.broadcast_arrays(item, i, j)
    ctr = np.stack([j >> one, i >> one, item, np.full(item.shape, offset & 0xFFFFFFFF, np.uint64)], axis=-1)
    key = np.array([seed & 0xFFFFFFFF, (seed >> 32) ^ (offset >> 32)], dtype=np.uint64)
    words = philox4x32_10(ctr, key)
    sel = ((i & one) * np.uint64(2) + (j & one)).astype(np.int64)
    w = np.take_along_axis(words, sel[..., None], axis=-1)[..., 0]
    kept = (w >> np.uint32(8)) >= np.uint32(dropout_threshold(p))
    return np.where(kept, inv_keep, np.float32(0.0)).astype(np.float32)


def keep_table(p: float, seed: int, offset: int, items: int, nq: int, nk: int) -> np.ndarray:
    """(items, nq, nk) float32: keep_scale over every item, query and key."""
    return keep_scale(p, seed, offset, np.arange(items)[:, None, None], np.arange(nq)[None, :, None],
                      np.arange(nk)[None, None, :])
