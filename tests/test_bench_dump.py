"""bench.py --dump-outputs: what lands in DIR for a given step result (host logic, no GPU)."""
import os

import numpy as np
import torch

import bench


def test_small_outputs_are_written_whole_in_float32_or_float64(tmp_path):
    a = torch.randn(50, 7)
    b = torch.randn(30, 3, dtype=torch.float64)
    h = torch.randn(20, 16).to(torch.bfloat16)
    bench.dump_outputs(str(tmp_path), {"a": a, "b": b, "h": h})
    assert sorted(os.listdir(tmp_path)) == ["a.npy", "b.npy", "h.npy"]
    ra, rb, rh = (np.load(tmp_path / f"{k}.npy") for k in "abh")
    assert ra.dtype == np.float32 and np.array_equal(ra, a.numpy())
    assert rb.dtype == np.float64 and np.array_equal(rb, b.numpy())
    assert rh.dtype == np.float32 and np.array_equal(rh, h.float().numpy())


def test_large_outputs_are_a_fixed_sample_of_rows_within_the_budget(tmp_path):
    x = torch.arange(4000 * 6, dtype=torch.float32).view(4000, 6)
    y = -x[:, :2]
    budget = 16 << 10
    for d in ("one", "two"):
        bench.dump_outputs(str(tmp_path / d), {"x": x, "y": y}, budget=budget)
    rx, ry = np.load(tmp_path / "one" / "x.npy"), np.load(tmp_path / "one" / "y.npy")
    assert rx.nbytes + ry.nbytes <= budget
    assert 0 < rx.shape[0] < 4000 and rx.shape[1] == 6 and ry.shape[1] == 2
    rows = (rx[:, 0] / 6).astype(np.int64)
    assert np.array_equal(rx, x.numpy()[rows]) and np.all(np.diff(rows) > 0)      # whole rows, sorted, no repeats
    assert np.array_equal(ry, y.numpy()[rows])                                    # equal row counts: the same rows
    for k in ("x", "y"):                                                           # same shapes: same sample
        assert np.array_equal(np.load(tmp_path / "one" / f"{k}.npy"), np.load(tmp_path / "two" / f"{k}.npy"))
