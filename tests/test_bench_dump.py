"""bench.py --dump-outputs: the planes it writes are float32, within the size limit, and the same rows on every run."""
import os

import numpy as np
import torch

import bench


def test_dump_planes_keeps_seeded_rows_within_budget(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    planes = np.arange(3 * 200 * 1000, dtype=np.float32).reshape(3, 200, 1000)
    bench.dump_planes(str(tmp_path), "np", planes)
    bench.dump_planes(str(tmp_path), "torch", torch.from_numpy(planes))
    bench.dump_planes(str(tmp_path), "half", planes, parts=2)
    bench.dump_planes(str(tmp_path), "small", planes[:, :10])
    a = np.load(tmp_path / "np.npy")
    assert a.dtype == np.float32 and a.shape[0] == 3 and a.shape[2] == 1000 and 0 < a.shape[1] < 200
    assert os.path.getsize(tmp_path / "np.npy") <= 1 << 20
    assert os.path.getsize(tmp_path / "half.npy") <= 1 << 19
    rows = (a[0, :, 0] / 1000).astype(np.int64)
    assert np.all(np.diff(rows) > 0)
    assert np.array_equal(a, planes[:, rows])
    assert np.array_equal(np.load(tmp_path / "torch.npy"), a)
    assert np.array_equal(np.load(tmp_path / "small.npy"), planes[:, :10])
