"""bench.py --dump-outputs: the files it writes for a SelectionVector (CPU tensors stand in for device ones)."""
import os

import numpy as np
import torch

import bench


def _load(d):
    return {f: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_short_vector_is_written_whole(tmp_path):
    """UINT32 entries above 2**31 (an int32 tensor on the device) come back as the row numbers they are."""
    rows = np.array([3, 7, 2**31 + 5, 2**32 - 1, 11], dtype=np.uint32)
    bench.dump_outputs(str(tmp_path), torch.from_numpy(rows.view(np.int32)), 4)
    got = _load(tmp_path)
    assert sorted(got) == ["selection_count.npy", "selection_vector.npy"]
    assert got["selection_count.npy"].dtype == np.float64 and got["selection_count.npy"].tolist() == [4.0]
    assert got["selection_vector.npy"].dtype == np.float64
    assert got["selection_vector.npy"].tolist() == [3.0, 7.0, 2.0**31 + 5, 2.0**32 - 1]


def test_long_vector_is_sampled_at_fixed_positions(tmp_path):
    n = 2 * bench.DUMP_SAMPLE + 1000
    vec = torch.arange(n, dtype=torch.int64) * 3 + 2**40
    a, b = tmp_path / "a", tmp_path / "b"
    bench.dump_outputs(str(a), vec, n)
    bench.dump_outputs(str(b), vec.clone(), n)
    got = _load(a)
    assert sorted(got) == ["selection_count.npy", "selection_positions.npy", "selection_vector.npy"]
    assert sum(os.path.getsize(os.path.join(a, f)) for f in got) <= 64 << 20
    pos = got["selection_positions.npy"]
    assert pos.size == bench.DUMP_SAMPLE and np.all(np.diff(pos) > 0) and pos[-1] < n
    assert np.array_equal(got["selection_vector.npy"], pos * 3 + 2.0**40)
    again = _load(b)
    assert all(np.array_equal(got[f], again[f]) for f in got)
    bench.dump_outputs(str(a), vec, 10)     # a later, shorter vector leaves no stale positions behind
    assert sorted(_load(a)) == ["selection_count.npy", "selection_vector.npy"]
