"""CPU-only: bench.py --dump-outputs writes float32 arrays, at fixed rows, within 64 MB for the default batch."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402


def test_dump_of_the_default_batch_is_sampled_exactly_and_fixed(tmp_path):
    n = 1 << bench.WORKLOADS["k256_varbase"][2]
    rng = np.random.default_rng(1)
    xy = rng.integers(0, 256, size=64 * n, dtype=np.uint8)
    inf = (rng.integers(0, 64, size=n) == 0).astype(np.uint8)
    names = bench.dump_outputs(str(tmp_path / "a"), "mul", n, xy, inf)
    bench.dump_outputs(str(tmp_path / "b"), "mul", n, xy, inf)
    assert names == ["index", "inf", "xy"]
    total = 0
    for name in names:
        a, b = (np.load(tmp_path / d / f"{name}.npy") for d in ("a", "b"))
        assert a.dtype == np.float32 and np.array_equal(a, b)
        total += os.path.getsize(tmp_path / "a" / f"{name}.npy")
    assert total <= 64 << 20
    idx = np.load(tmp_path / "a" / "index.npy").astype(np.int64)
    assert len(idx) == bench.DUMP_ROWS and np.all(np.diff(idx) > 0)
    assert np.array_equal(np.load(tmp_path / "a" / "xy.npy"), xy.reshape(n, 64)[idx].astype(np.float32))
    assert np.array_equal(np.load(tmp_path / "a" / "inf.npy"), inf[idx].astype(np.float32))


def test_small_batches_and_other_ops_are_dumped_whole(tmp_path):
    n = 300
    v = np.arange(n, dtype=np.uint8)
    assert bench.dump_outputs(str(tmp_path / "s"), "schnorr", n, v, np.zeros(n, np.uint8)) == ["index", "valid"]
    assert np.array_equal(np.load(tmp_path / "s" / "valid.npy"), v.astype(np.float32))
    xy = np.arange(64, dtype=np.uint8)
    assert bench.dump_outputs(str(tmp_path / "l"), "lincomb", n, xy, np.ones(1, np.uint8)) == ["inf", "xy"]
    assert np.load(tmp_path / "l" / "xy.npy").shape == (1, 64)
