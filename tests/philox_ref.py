"""numpy restatement of the attention-dropout keep rule (rgb-experiment_b200/csrc/philox.cuh), the arbiter the
device mask and the fused kernels are checked against.

For edge e and head h:  u = Philox4x32-10(counter (e, h, 0, 0), key (seed & 0xffffffff, seed >> 32)).word0;
the edge is dropped iff u < floor(p * 2^32); a kept edge is multiplied by float32(1 / (1 - p)), a dropped one by 0.
"""
import math

import numpy as np

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = 0x9E3779B9, 0xBB67AE85
MASK32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """ctr: four uint32 arrays (broadcastable), key: two ints -> the four output words as uint32 arrays."""
    c0, c1, c2, c3 = (np.asarray(c, dtype=np.uint64) & MASK32 for c in ctr)
    k0, k1 = int(key[0]) & 0xFFFFFFFF, int(key[1]) & 0xFFFFFFFF
    for _ in range(10):
        p0 = M0 * c0
        p1 = M1 * c2
        hi0, lo0 = p0 >> np.uint64(32), p0 & MASK32
        hi1, lo1 = p1 >> np.uint64(32), p1 & MASK32
        c0, c1, c2, c3 = hi1 ^ c1 ^ np.uint64(k0), lo1, hi0 ^ c3 ^ np.uint64(k1), lo0
        k0, k1 = (k0 + W0) & 0xFFFFFFFF, (k1 + W1) & 0xFFFFFFFF
    return tuple(c.astype(np.uint32) for c in (c0, c1, c2, c3))


def seed_key(seed: int):
    s = int(seed) & 0xFFFFFFFFFFFFFFFF
    return s & 0xFFFFFFFF, s >> 32


def bits(seed: int, e, h):
    e, h = np.broadcast_arrays(np.asarray(e, dtype=np.uint64), np.asarray(h, dtype=np.uint64))
    z = np.zeros_like(e)
    return philox4x32_10((e, h, z, z), seed_key(seed))[0]


def thresh(p: float) -> int:
    return int(math.floor(p * 4294967296.0))


def keep(seed: int, e, h, p: float):
    u = bits(seed, e, h).astype(np.uint64)
    return u >= np.uint64(thresh(p))          # p == 1: thresh = 2^32, nothing is kept


def mask(seed: int, nnz: int, H: int, p: float) -> np.ndarray:
    """[nnz, H] float32 multipliers in edge order."""
    e = np.arange(nnz, dtype=np.uint64)[:, None]
    h = np.arange(H, dtype=np.uint64)[None, :]
    k = keep(seed, e, h, p)
    scale = np.float32(1.0 / (1.0 - p)) if p < 1.0 else np.float32(0.0)
    return np.where(k, scale, np.float32(0.0)).astype(np.float32)
