"""numpy restatement of SuperGAT's device sampling (rgb-experiment_b200/csrc/philox.cuh, csrc/supergat_loss.cu), the
arbiter the device keep mask and negatives are checked against.

  positive edge e kept iff thresh == 0 or Philox4x32-10(counter (e, 0, 1, 0), key (seed lo, seed hi)).word0 >= thresh,
      thresh = floor((1 - edge_sample_ratio) * 2^32)
  negative candidate k of round r: (w0, w1, w2, w3) = Philox4x32-10(counter (k, r, 2, 0), key),
      row = (w1:w0 * N) >> 64, col = (w3:w2 * N) >> 64; rejected iff (row, col) is a pair of U
  survivors of rounds 0, 1, 2 concatenated in (round, k) order until there are num_neg, then cut to num_neg -- the
  loop of torch_geometric's negative_sampling, with (num_neg, sample_size) from its float formulas.
"""
import math

import numpy as np

import philox_ref as PR

U32 = np.uint64(0xFFFFFFFF)


def keep_thresh(edge_sample_ratio: float) -> int:
    return int(math.floor((1.0 - float(edge_sample_ratio)) * 4294967296.0))


def edge_sample_bits(seed: int, e) -> np.ndarray:
    e = np.asarray(e, dtype=np.uint64)
    z = np.zeros_like(e)
    return PR.philox4x32_10((e, z, z + np.uint64(1), z), PR.seed_key(seed))[0]


def keep_mask(seed: int, nnz: int, edge_sample_ratio: float) -> np.ndarray:
    t = keep_thresh(edge_sample_ratio)
    if t == 0:
        return np.ones(nnz, dtype=bool)
    return edge_sample_bits(seed, np.arange(nnz, dtype=np.uint64)).astype(np.uint64) >= np.uint64(t)


def umulhi64(lo, hi, n: int) -> np.ndarray:
    """((hi:lo) * n) >> 64 for 32-bit words lo, hi and n < 2^31, without overflowing uint64."""
    lo, hi, n = lo.astype(np.uint64), hi.astype(np.uint64), np.uint64(n)
    return (hi * n + ((lo * n) >> np.uint64(32))) >> np.uint64(32)


def candidates(seed: int, rnd: int, S: int, N: int):
    k = np.arange(S, dtype=np.uint64)
    z = np.zeros_like(k)
    w0, w1, w2, w3 = PR.philox4x32_10((k, z + np.uint64(rnd), z + np.uint64(2), z), PR.seed_key(seed))
    return umulhi64(w0, w1, N).astype(np.int64), umulhi64(w2, w3, N).astype(np.int64)


def neg_counts(N: int, E_u: int, num_neg_samples: int):
    """(num_neg, sample_size) as negative_sampling computes them from E_u = edge_index.size(1)."""
    size = N * N
    num_neg = min(int(num_neg_samples), size - E_u)
    if num_neg <= 0:
        return num_neg, 0
    alpha = abs(1 / (1 - 1.1 * (E_u / size)))
    return num_neg, int(alpha * num_neg)


def undirected_keys(src, dst, N: int, symmetrize: bool = True) -> np.ndarray:
    src, dst = np.asarray(src, dtype=np.int64), np.asarray(dst, dtype=np.int64)
    if symmetrize:
        src, dst = np.concatenate([src, dst]), np.concatenate([dst, src])
    return np.unique(src * N + dst)


def negatives(seed: int, N: int, u_keys: np.ndarray, num_neg: int, S: int):
    """(src, dst, rounds run) of the sampler."""
    if num_neg <= 0 or S <= 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int64), 0
    rows, cols = [], []
    have = 0
    for r in range(3):
        row, col = candidates(seed, r, S, N)
        ok = ~np.isin(row * N + col, u_keys)
        rows.append(row[ok])
        cols.append(col[ok])
        have += int(ok.sum())
        if have >= num_neg:
            break
    row, col = np.concatenate(rows)[:num_neg], np.concatenate(cols)[:num_neg]
    return row, col, r + 1
