"""bench.py --dump-outputs (host side, no GPU): within the size budget the torques are written whole; beyond it, a fixed
sample of robots whose indices are written beside them, identical from call to call."""
import os

import numpy as np

import bench


def _dump(tmp_path, name, tau):
    out = str(tmp_path / name)
    bench.dump_outputs(out, tau)
    files = sorted(os.listdir(out))
    return out, files, sum(os.path.getsize(os.path.join(out, f)) for f in files)


def test_dump_within_budget_is_the_whole_array(tmp_path):
    tau = np.random.default_rng(1).standard_normal((7, 1000))
    out, files, _ = _dump(tmp_path, "whole", tau)
    assert files == ["tau.npy"]
    got = np.load(os.path.join(out, "tau.npy"))
    assert got.dtype == np.float64 and np.array_equal(got, tau)


def test_dump_beyond_budget_is_a_fixed_sample(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES_MAX", 40_000)
    tau = np.random.default_rng(2).standard_normal((7, 5000))      # 280 kB of torques
    runs = []
    for name in ("a", "b"):
        out, files, size = _dump(tmp_path, name, tau)
        assert files == ["robot_index.npy", "tau.npy"] and size <= bench.DUMP_BYTES_MAX
        idx = np.load(os.path.join(out, "robot_index.npy"))
        got = np.load(os.path.join(out, "tau.npy"))
        assert idx.dtype == np.float64 and got.dtype == np.float64
        i = idx.astype(np.int64)
        assert np.array_equal(i, idx) and (np.diff(i) > 0).all() and 0 <= i[0] and i[-1] < tau.shape[1]
        assert got.shape == (7, i.size) and i.size > 0.9 * (bench.DUMP_BYTES_MAX - 4096) / 8 / 8
        assert np.array_equal(got, tau[:, i])
        runs.append((idx, got))
    assert np.array_equal(runs[0][0], runs[1][0]) and np.array_equal(runs[0][1], runs[1][1])
