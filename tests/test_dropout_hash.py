"""The attention-dropout keep rule on the CPU: the numpy restatement (philox_ref) reproduces the Random123
known-answer vectors of Philox4x32-10, and the device header csrc/philox.cuh, compiled as host code, gives the same
words and the same multipliers on a grid of (seed, edge, head, p)."""
import os
import shutil
import subprocess

import numpy as np
import pytest

import philox_ref as PR

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "rgb-experiment_b200", "csrc")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")

# Random123 kat_vectors: philox4x32_10 (counter, key) -> output
KAT = [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
]
SEEDS = [0, 1, 0x0123456789ABCDEF, 0x7FFFFFFFFFFFFFFF, 0xFFFFFFFF00000001]
PS = [0.5, 0.1, 0.2, 0.3, 1.0 - 2.0 ** -24, 1.0]
NE, NH = 257, 8


@pytest.mark.parametrize("ctr,key,want", KAT)
def test_numpy_philox_reproduces_known_answers(ctr, key, want):
    got = PR.philox4x32_10(tuple(np.array([c], dtype=np.uint64) for c in ctr), key)
    assert tuple(int(w[0]) for w in got) == want


def test_numpy_keep_rule_edges():
    e = np.arange(100_000, dtype=np.uint64)
    assert PR.keep(5, e, 0, 0.0).all()
    assert not PR.keep(5, e, 0, 1.0).any()
    frac = PR.keep(5, e, 3, 0.5).mean()
    assert abs(frac - 0.5) < 5 * (0.25 / e.size) ** 0.5
    m = PR.mask(9, 1000, 3, 0.2)
    assert set(np.unique(m).tolist()) <= {0.0, float(np.float32(1.0 / 0.8))}


HOST_PROGRAM = r"""
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "philox.cuh"
using namespace rgbmp;
int main(int argc, char** argv) {
  // mode 0: ctr0 ctr1 ctr2 ctr3 key0 key1 -> four words
  // mode 1: seed n_e n_h thresh scale   -> for every (e, h): bits and the multiplier's float bits
  if (atoi(argv[1]) == 0) {
    uint32_t c[4], o[4];
    for (int i = 0; i < 4; ++i) c[i] = (uint32_t)strtoul(argv[2 + i], 0, 0);
    PhiloxKey k{(uint32_t)strtoul(argv[6], 0, 0), (uint32_t)strtoul(argv[7], 0, 0)};
    philox4x32_10(c, k, o);
    printf("%08x %08x %08x %08x\n", o[0], o[1], o[2], o[3]);
    return 0;
  }
  const PhiloxKey k = philox_key(strtoull(argv[2], 0, 0));
  const int ne = atoi(argv[3]), nh = atoi(argv[4]);
  const uint32_t thresh = (uint32_t)strtoul(argv[5], 0, 0);
  const float scale = strtof(argv[6], 0);
  for (int e = 0; e < ne; ++e)
    for (int h = 0; h < nh; ++h) {
      const float m = dropout_mult(k, (uint32_t)e, (uint32_t)h, thresh, scale);
      uint32_t mb;
      memcpy(&mb, &m, 4);
      printf("%u %u\n", dropout_bits(k, (uint32_t)e, (uint32_t)h), mb);
    }
  return 0;
}
"""


@pytest.fixture(scope="module")
def host_prog(tmp_path_factory):
    if not os.path.exists(NVCC) and shutil.which("nvcc") is None:
        pytest.skip("nvcc is not available")
    nvcc = NVCC if os.path.exists(NVCC) else shutil.which("nvcc")
    d = tmp_path_factory.mktemp("philox_host")
    src = d / "philox_host.cu"
    src.write_text(HOST_PROGRAM)
    exe = d / "philox_host"
    r = subprocess.run([nvcc, "-O2", "-std=c++17", "-I", CSRC, str(src), "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return str(exe)


def _abi_params(p):
    """what ops._dropout_struct passes: p == 1 -> thresh 2^32 - 1 and scale 0"""
    if p >= 1.0:
        return 0xFFFFFFFF, 0.0
    return PR.thresh(p), float(np.float32(1.0 / (1.0 - p)))


@pytest.mark.parametrize("ctr,key,want", KAT)
def test_device_header_as_host_code_reproduces_known_answers(host_prog, ctr, key, want):
    out = subprocess.run([host_prog, "0", *map(str, ctr), *map(str, key)], capture_output=True, text=True, check=True)
    assert tuple(int(w, 16) for w in out.stdout.split()) == want


@pytest.mark.parametrize("seed", SEEDS)
def test_device_header_matches_numpy_keep_rule(host_prog, seed):
    e = np.arange(NE, dtype=np.uint64)[:, None]
    h = np.arange(NH, dtype=np.uint64)[None, :]
    want_bits = PR.bits(seed, e, h).reshape(-1)
    for p in PS:
        thresh, scale = _abi_params(p)
        out = subprocess.run([host_prog, "1", str(seed), str(NE), str(NH), str(thresh), repr(scale)],
                             capture_output=True, text=True, check=True)
        got = np.array([ln.split() for ln in out.stdout.splitlines()], dtype=np.uint64)
        assert np.array_equal(got[:, 0].astype(np.uint32), want_bits), (seed, p)
        want_mask = PR.mask(seed, NE, NH, p).reshape(-1)
        assert np.array_equal(got[:, 1].astype(np.uint32), want_mask.view(np.uint32)), (seed, p)
        kept = got[:, 1] != 0
        if p < 1.0:
            assert np.array_equal(kept, PR.keep(seed, e, h, p).reshape(-1)), (seed, p)
