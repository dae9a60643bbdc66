"""bench.py --dump-outputs: float32 .npy files, whole tensors under the 64 MiB budget, a fixed seeded row sample above it."""
import numpy as np
import torch

import bench


def test_dump_writes_float32_whole_tensor(tmp_path):
    x = torch.randn(4, 3, 8, dtype=torch.float64)
    bench.dump_output(str(tmp_path / "d"), "encoder_output", x)
    got = np.load(tmp_path / "d" / "encoder_output.npy")
    assert got.dtype == np.float32 and np.array_equal(got, x.float().numpy())


def test_dump_samples_rows_over_budget_deterministically(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BUDGET_BYTES", 10 * 16 * 4)
    x = torch.arange(100 * 16, dtype=torch.float32).view(100, 16)
    bench.dump_output(str(tmp_path / "a"), "encoder_output", x)
    bench.dump_output(str(tmp_path / "b"), "encoder_output", x)
    a, b = np.load(tmp_path / "a" / "encoder_output.npy"), np.load(tmp_path / "b" / "encoder_output.npy")
    assert a.shape == (10, 16) and np.array_equal(a, b)
    rows = a[:, 0] / 16
    assert np.all(np.diff(rows) > 0) and np.array_equal(a, x.numpy()[rows.astype(int)])
