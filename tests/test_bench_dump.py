"""bench.py --dump-outputs: the size budget, whole small arrays, and the same seeded sample from run to run.  CPU only."""
import os

import numpy as np
import torch

import bench


def test_dump_outputs_stays_in_budget_and_is_reproducible(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 32 << 10)   # small enough to stay off torch's CPU thread pool
    g = torch.Generator().manual_seed(0)
    arrays = {"loss": torch.tensor(1.5, dtype=torch.float64), "grad.small": torch.randn(7, 3, generator=g),
              "grad.big": torch.randn(128, 128, generator=g)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(k + ".npy" for k in arrays)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 32 << 10
    assert np.load(tmp_path / "a" / "loss.npy").dtype == np.float64
    assert np.array_equal(np.load(tmp_path / "a" / "grad.small.npy"), arrays["grad.small"].numpy())
    big = np.load(tmp_path / "a" / "grad.big.npy")
    assert big.dtype == np.float32 and 0 < big.size < arrays["grad.big"].numel()
    assert np.isin(big, arrays["grad.big"].numpy()).all()
    for f in files:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))
