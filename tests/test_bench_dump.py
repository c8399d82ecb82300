"""CPU: the format of `bench.py --dump-outputs` (bench.dump_outputs) on host tensors — every sampled 64-bit word comes back
exactly from its two float64 halves, the sample positions depend only on the array's size, and the default workload's
dump stays under 64 MB."""
import os

import numpy as np

import bench


def _words(n, seed):
    return np.random.default_rng(seed).integers(0, 2**64, size=n, dtype=np.uint64)


def _dump(tmp, root, arrays):
    import torch
    bench.dump_outputs(str(tmp), root, {k: torch.from_numpy(v.view(np.int64)) for k, v in arrays.items()})
    return {f[:-4]: np.load(os.path.join(tmp, f)) for f in os.listdir(tmp)}


def _rebuild(halves):
    assert halves.dtype == np.float64 and halves.shape[1] == 2
    lo, hi = halves[:, 0].astype(np.uint64), halves[:, 1].astype(np.uint64)
    return lo | (hi << np.uint64(32))


def test_dump_is_exact_and_reproducible(tmp_path):
    small = _words(1000, 1)
    big = _words(5 * (bench.DUMP_SAMPLE // 4 + 123), 2).reshape(5, -1)
    root = bytes(range(32))
    got = _dump(tmp_path / "a", root, {"small": small, "big": big})
    assert got["merkle_root"].tolist() == list(range(32))
    assert np.array_equal(_rebuild(got["small"]), small)
    assert np.array_equal(got["small_index"], np.arange(1000))
    idx = got["big_index"].astype(np.int64)
    assert len(idx) == bench.DUMP_SAMPLE and np.all(np.diff(idx) > 0) and idx[-1] < big.size
    assert np.array_equal(_rebuild(got["big"]), big.reshape(-1)[idx])
    again = _dump(tmp_path / "b", root, {"big": _words(big.size, 3)})
    assert np.array_equal(again["big_index"], got["big_index"])


def test_default_workload_dump_fits_64_mb():
    per_array = bench.DUMP_SAMPLE * (2 * 8 + 8)        # halves + index, float64
    assert 3 * per_array + 32 * 8 < 64 << 20
