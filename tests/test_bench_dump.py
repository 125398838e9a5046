"""bench.py --dump-outputs: float32 .npy files, at most the byte budget in all, the same seeded rows in every per-simplex array."""
import os
import sys

import numpy as np
import torch

from conftest import ROOT

if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import bench


def _dump(path, budget):
    y = torch.arange(1000 * 6, dtype=torch.float64).reshape(1000, 2, 3)
    bench.dump_outputs(str(path), {"y": y, "grad_h": -y}, {"grad.w": torch.ones(4, 5)}, budget=budget)
    return {f[:-4]: np.load(os.path.join(path, f)) for f in sorted(os.listdir(path))}


def test_dump_outputs_whole_when_under_budget(tmp_path):
    out = _dump(tmp_path, 1 << 20)
    assert sorted(out) == ["grad.w", "grad_h", "y"]
    assert all(a.dtype == np.float32 for a in out.values())
    assert out["y"].shape == (1000, 2, 3) and np.array_equal(out["grad_h"], -out["y"])


def test_dump_outputs_samples_rows_over_budget(tmp_path):
    budget = 20000
    out = _dump(tmp_path / "a", budget)
    assert sum(os.path.getsize(os.path.join(tmp_path / "a", f)) for f in os.listdir(tmp_path / "a")) <= budget
    assert out["grad.w"].shape == (4, 5)
    n = out["y"].shape[0]
    assert 0 < n < 1000 and out["y"].shape[1:] == (2, 3)
    rows = out["y"][:, 0, 0] / 6
    assert np.array_equal(rows, np.sort(rows)) and np.array_equal(out["grad_h"], -out["y"])
    again = _dump(tmp_path / "b", budget)
    assert all(np.array_equal(out[k], again[k]) for k in out)
