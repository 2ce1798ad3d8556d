"""SuperGAT's device sampling on the CPU: the numpy restatement (supergat_sampling_ref) computes negative_sampling's
(num_neg, sample_size) exactly as the oracle does and reproduces the oracle's round loop when fed the same candidate
stream; the helpers of csrc/philox.cuh, compiled as host code, give the same words, rows and columns as numpy; the
C ABI reports argument errors without a GPU."""
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

import supergat_sampling_ref as SR
from oracle import layers as OL

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "rgb-experiment_b200", "csrc")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
SEEDS = [0, 1, 0x0123456789ABCDEF, 0x7FFFFFFFFFFFFFFF, 0xFFFFFFFF00000001]


def _edges(N, E, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(N, (2, E), generator=g)


def _free_key(ei, N):
    keys = set((ei[0] * N + ei[1]).tolist())
    return next(k for k in range(N * N) if k not in keys)


@pytest.mark.parametrize("N,E_u", [(5, 7), (5, 20), (5, 24), (5, 25), (5, 31), (50, 400), (300, 5000), (1000, 2),
                                   (70_000, 100_000), (20, 398)])
@pytest.mark.parametrize("ratio", [0.5, 1.0, 0.25, 3.0])
def test_counts_agree_with_oracle_negative_sampling(monkeypatch, N, E_u, ratio):
    ei = _edges(N, E_u, N + E_u)
    want_num = int(ratio * E_u)
    seen = []
    fill = _free_key(ei, N) if E_u < N * N else 0
    real_randint = torch.randint

    def fake_randint(high, size, **kw):
        seen.append((high, size))
        return torch.full(size, fill, dtype=torch.long)          # every candidate survives round 0

    monkeypatch.setattr(torch, "randint", fake_randint)
    out = OL.negative_sampling(ei, N, want_num)
    monkeypatch.setattr(torch, "randint", real_randint)
    num_neg, S = SR.neg_counts(N, E_u, want_num)
    if num_neg <= 0:
        assert out.size(1) == 0 and not seen
        return
    assert seen == [(N * N, (S,))]
    assert out.size(1) == num_neg


@pytest.mark.parametrize("case", [(5, 17, 6, 0), (20, 398, 2, 1), (300, 5000, 2500, 2), (50, 400, 800, 3)])
@pytest.mark.parametrize("seed", SEEDS[:3])
def test_restatement_is_the_oracle_loop_on_the_same_candidates(monkeypatch, case, seed):
    """Fed this restatement's candidates of rounds 0, 1, 2, the oracle's loop-with-break returns exactly its negatives."""
    N, E, want, gseed = case
    ei = _edges(N, E, gseed)
    keys = SR.undirected_keys(ei[0].numpy(), ei[1].numpy(), N, symmetrize=False)
    num_neg, S = SR.neg_counts(N, E, want)
    rounds = iter(range(3))

    def fake_randint(high, size, **kw):
        row, col = SR.candidates(seed, next(rounds), size[0], N)
        return torch.from_numpy(row * N + col)

    monkeypatch.setattr(torch, "randint", fake_randint)
    out = OL.negative_sampling(ei, N, want)
    monkeypatch.undo()
    row, col, _ = SR.negatives(seed, N, keys, num_neg, S)
    assert np.array_equal(out[0].numpy(), row) and np.array_equal(out[1].numpy(), col)


def test_keep_rule_and_candidate_range():
    e = np.arange(200_000, dtype=np.uint64)
    assert SR.keep_mask(3, e.size, 1.0).all()
    assert not SR.keep_mask(3, e.size, 0.0).any()
    frac = SR.keep_mask(3, e.size, 0.7).mean()
    assert abs(frac - 0.7) < 5 * (0.21 / e.size) ** 0.5
    for N in (1, 2, 7, 1000, (1 << 31) - 1):
        row, col = SR.candidates(9, 1, 5000, N)
        assert row.min() >= 0 and row.max() < N and col.min() >= 0 and col.max() < N
    row, _ = SR.candidates(9, 0, 200_000, 10)
    assert np.abs(np.bincount(row, minlength=10) / row.size - 0.1).max() < 0.005


HOST_PROGRAM = r"""
#include <stdio.h>
#include <stdlib.h>
#include "philox.cuh"
using namespace rgbmp;
int main(int argc, char** argv) {
  // seed n round N -> for k < n: edge_sample_bits(k) row col
  const PhiloxKey key = philox_key(strtoull(argv[1], 0, 0));
  const int n = atoi(argv[2]);
  const uint32_t round = (uint32_t)atoi(argv[3]);
  const uint64_t N = strtoull(argv[4], 0, 0);
  for (int k = 0; k < n; ++k) {
    uint32_t row, col;
    neg_candidate(key, (uint32_t)k, round, N, row, col);
    printf("%u %u %u\n", edge_sample_bits(key, (uint32_t)k), row, col);
  }
  return 0;
}
"""


@pytest.fixture(scope="module")
def host_prog(tmp_path_factory):
    if not os.path.exists(NVCC) and shutil.which("nvcc") is None:
        pytest.skip("nvcc is not available")
    nvcc = NVCC if os.path.exists(NVCC) else shutil.which("nvcc")
    d = tmp_path_factory.mktemp("sgat_host")
    src = d / "sgat_host.cu"
    src.write_text(HOST_PROGRAM)
    exe = d / "sgat_host"
    r = subprocess.run([nvcc, "-O2", "-std=c++17", "-I", CSRC, str(src), "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return str(exe)


@pytest.mark.parametrize("seed", SEEDS)
@pytest.mark.parametrize("rnd,N", [(0, 5), (1, 300), (2, (1 << 31) - 1)])
def test_device_header_matches_numpy(host_prog, seed, rnd, N):
    n = 513
    out = subprocess.run([host_prog, str(seed), str(n), str(rnd), str(N)], capture_output=True, text=True, check=True)
    got = np.array([ln.split() for ln in out.stdout.splitlines()], dtype=np.int64)
    assert np.array_equal(got[:, 0], SR.edge_sample_bits(seed, np.arange(n)).astype(np.int64))
    row, col = SR.candidates(seed, rnd, n, N)
    assert np.array_equal(got[:, 1], row) and np.array_equal(got[:, 2], col)


def test_cabi_argument_errors_do_not_need_a_gpu():
    import ctypes as C
    import rgb_experiment_b200 as R
    L = R._lib.lib()
    assert L.rgbmp_sgat_negative_sampling(None, None, 5, None, 3, 10, None, None, None, None, 0, 0, None) == R._lib.EINVAL
    s = R._lib.SgatSampleStruct(8, None, None, 0)               # any non-NULL seed pointer: nothing is launched
    cnt = 8
    rc = L.rgbmp_sgat_negative_sampling(8, 8, 5, C.byref(s), 3, 1 << 31, 8, 8, cnt, 8, 1 << 40, 0, None)
    assert rc == R._lib.ERANGE
    assert b"sample_size" in L.rgbmp_last_error()
    bad = R._lib.SgatSampleStruct(8, None, None, (1 << 32) + 1)
    assert L.rgbmp_sgat_keep_mask(C.byref(bad), 10, 8, 0, None) == R._lib.EINVAL
    assert L.rgbmp_sgat_loss_forward(None, None, None, None, 0, 8, 1.0, None, None, None, 0, 0, None) == R._lib.EINVAL
    assert L.rgbmp_sgat_loss_workspace_bytes(1000) > 8000
