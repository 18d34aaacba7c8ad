"""Dropout masks of the training step, restated in numpy -- TEST INFRASTRUCTURE.

An independent statement of the contract the kernels implement (internnav_b200/csrc/dropout.cuh): Philox4x32-10
(Salmon, Moraes, Dror, Shaw, "Parallel random numbers: as easy as 1, 2, 3", SC 2011) with key (seed_lo, seed_hi) and
counter (e >> 2 low word, high word, site | rank << 16, step); element e of the site's row-major tensor is dropped iff
output word e & 3 is below floor(p * 2^32); kept elements are scaled by float32(1 / (1 - p)).
"""
import math

import numpy as np

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = 0x9E3779B9, 0xBB67AE85
_LO = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """ctr: uint32 [..., 4], key: (k0, k1) -> uint32 [..., 4]."""
    c = [np.asarray(ctr[..., i], dtype=np.uint64) for i in range(4)]
    k0, k1 = int(key[0]) & 0xFFFFFFFF, int(key[1]) & 0xFFFFFFFF
    for r in range(10):
        if r:
            k0, k1 = (k0 + _W0) & 0xFFFFFFFF, (k1 + _W1) & 0xFFFFFFFF
        p0, p1 = _M0 * c[0], _M1 * c[2]
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & _LO, p1 >> np.uint64(32), p1 & _LO
        c = [hi1 ^ c[1] ^ np.uint64(k0), lo1, hi0 ^ c[3] ^ np.uint64(k1), lo0]
    return np.stack(c, axis=-1).astype(np.uint32)


def threshold(p):
    return int(math.floor(float(p) * 4294967296.0))


def scale(p):
    return np.float32(1.0 / (1.0 - float(p)))


def words(n, seed, site, step=0, rank=0):
    """The Philox word deciding each of elements 0 .. n-1 (uint32 [n])."""
    g = np.arange((n + 3) // 4, dtype=np.uint64)
    ctr = np.empty((g.size, 4), dtype=np.uint64)
    ctr[:, 0], ctr[:, 1] = g & _LO, g >> np.uint64(32)
    ctr[:, 2] = (int(site) | (int(rank) << 16)) & 0xFFFFFFFF
    ctr[:, 3] = int(step) & 0xFFFFFFFF
    seed = int(seed)
    return philox4x32_10(ctr, (seed & 0xFFFFFFFF, seed >> 32)).reshape(-1)[:n]


def keep_mask(shape, seed, site, p, step=0, rank=0):
    """bool [shape]: True where the element is kept."""
    n = int(np.prod(shape))
    return (words(n, seed, site, step, rank) >= np.uint32(threshold(p))).reshape(shape)


def multiplier(shape, seed, site, p, step=0, rank=0):
    """float32 [shape]: 0 where dropped, float32(1 / (1 - p)) where kept (the factor the kernels apply)."""
    return keep_mask(shape, seed, site, p, step, rank).astype(np.float32) * scale(p)
