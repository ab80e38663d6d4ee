"""bench.py --dump-outputs without a device: the file written for one workload."""
import numpy as np

import bench


def test_dump_outputs_is_a_fixed_sample(tmp_path):
    rng = np.random.default_rng(1)
    arrays = [rng.integers(0, 256, n, dtype=np.uint8) for n in (5000, 7, 123457)]
    bench.dump_outputs(str(tmp_path / "a"), "w", arrays)
    bench.dump_outputs(str(tmp_path / "b"), "w", [a.copy() for a in arrays])
    got = np.load(tmp_path / "a" / "w.npy")
    assert got.dtype == np.float32 and got.shape == (3, bench.DUMP_VALUES // 3)
    assert 6 * got.nbytes <= 64 << 20  # six workloads per run
    assert np.array_equal(got, np.load(tmp_path / "b" / "w.npy"))  # same outputs, same file
    for row, src in zip(got, arrays):
        assert set(row.astype(np.uint8).tolist()) <= set(src.tolist())
    assert set(got[1].astype(np.uint8).tolist()) == set(arrays[1].tolist())
    bench.dump_outputs(str(tmp_path / "c"), "w", [arrays[0] ^ 0xFF] + arrays[1:])
    changed = np.load(tmp_path / "c" / "w.npy")
    assert np.array_equal(changed[0], 255 - got[0]) and np.array_equal(changed[1:], got[1:])
