"""bench.py --dump-outputs: the file it writes (CPU only: the helper is fed a host array)."""
import os

import numpy as np

import bench


def test_dump_is_the_whole_output_when_it_fits(tmp_path):
    d = np.random.default_rng(0).random(1000) * 300
    bench.dump_outputs(str(tmp_path), d)
    got = np.load(os.path.join(str(tmp_path), "distances.npy"))
    assert got.dtype == np.float64 and np.array_equal(got, d)


def test_dump_of_a_large_output_is_a_fixed_sample_in_pair_order(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 800)
    d = np.arange(10_000, dtype=np.float64)
    bench.dump_outputs(str(tmp_path / "a"), d)
    bench.dump_outputs(str(tmp_path / "b"), d)
    a = np.load(str(tmp_path / "a" / "distances.npy"))
    b = np.load(str(tmp_path / "b" / "distances.npy"))
    assert a.shape == (100,) and np.array_equal(a, b)
    assert np.all(np.diff(a) > 0) and np.all(np.isin(a, d))


def test_dump_budget_stays_under_64_mb():
    assert bench.DUMP_BYTES + 4096 <= 64_000_000
