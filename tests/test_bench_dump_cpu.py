"""CPU: what `bench.py --dump-outputs DIR` writes -- float32 images, within its size limit, the same subset every run."""
import numpy as np
import torch

import bench


def test_dump_samples_writes_the_whole_batch_as_float32(tmp_path):
    x = torch.randn(8, 3, 16, 16, dtype=torch.float64)
    bench.dump_samples(str(tmp_path / "out"), x)
    got = np.load(tmp_path / "out" / "samples.npy")
    assert got.dtype == np.float32
    assert np.array_equal(got, x.float().numpy())


def test_dump_samples_keeps_a_fixed_subset_of_whole_images(tmp_path, monkeypatch):
    per_image = 3 * 16 * 16
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 10 * per_image * 4)
    x = torch.arange(25 * per_image, dtype=torch.float32).reshape(25, 3, 16, 16)
    for d in ("a", "b"):
        bench.dump_samples(str(tmp_path / d), x)
    a, b = np.load(tmp_path / "a" / "samples.npy"), np.load(tmp_path / "b" / "samples.npy")
    assert a.shape == (10, 3, 16, 16) and a.nbytes <= bench.DUMP_MAX_BYTES
    assert np.array_equal(a, b)
    rows = (a[:, 0, 0, 0] / per_image).astype(int)
    assert list(rows) == sorted(set(rows)) and rows.max() < 25
    assert np.array_equal(a, x.numpy()[rows])
