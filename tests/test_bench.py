"""CPU: bench.py --dump-outputs writes float32 .npy files under 64 MB, the same rows on every run."""
import os

import numpy as np

import bench


def test_dump_outputs_is_float32_capped_and_deterministic(tmp_path):
    small = np.arange(12, dtype=np.float64).reshape(3, 4)
    bench.dump_outputs(str(tmp_path / "a"), "small", small)
    back = np.load(tmp_path / "a" / "small.npy")
    assert back.dtype == np.float32 and np.array_equal(back, small)

    big = np.random.default_rng(1).standard_normal((40000, 500)).astype(np.float32)     # 80 MB
    big[:, 0] = np.arange(len(big))                                                     # row ids
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), "big", big)
    path = tmp_path / "a" / "big.npy"
    assert os.path.getsize(path) <= 64 * 10 ** 6
    a, b = np.load(path), np.load(tmp_path / "b" / "big.npy")
    assert a.dtype == np.float32 and a.shape[1] == 500 and np.array_equal(a, b)
    # a sample of whole rows of the output, in their original order
    rows = a[:, 0].astype(np.int64)
    assert np.all(np.diff(rows) > 0) and np.array_equal(big[rows], a)
