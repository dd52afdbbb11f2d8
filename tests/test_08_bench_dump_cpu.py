"""bench.py --dump-outputs writer: dtypes, the seeded sample of large outputs and the size budget (no GPU)."""
import os

import numpy as np
import pytest
import torch

import bench


def test_dump_outputs_dtypes_and_sample(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 1000)
    big = torch.arange(5000, dtype=torch.float32)
    arrays = {"a.ints": np.array([2 ** 31 - 1, -5], np.int32), "a.half": torch.tensor([0.5], dtype=torch.float16),
              "a.f64": np.array([1 / 3]), "a.flags": torch.tensor([True, False]), "a.scalar": 1.25, "big": big}
    for d in ("x", "y"):
        bench.dump_outputs(arrays, str(tmp_path / d))
    got = {f[:-4]: np.load(tmp_path / "x" / f) for f in os.listdir(tmp_path / "x")}
    assert set(got) == set(arrays)
    assert got["a.ints"].dtype == np.float64 and got["a.ints"].tolist() == [2 ** 31 - 1, -5]
    assert got["a.half"].dtype == np.float32 and got["a.f64"].dtype == np.float64 and got["a.flags"].tolist() == [1.0, 0.0]
    s = got["big"]
    assert s.dtype == np.float32 and s.shape == (1000,) and len(np.unique(s)) == 1000 and (np.diff(s) > 0).all()
    np.testing.assert_array_equal(s, np.load(tmp_path / "y" / "big.npy"))        # same indices on every run


def test_dump_outputs_refuses_more_than_the_budget(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_BUDGET", 1000)
    with pytest.raises(SystemExit):
        bench.dump_outputs({"x": np.zeros(1000, np.float32)}, str(tmp_path / "d"))
    assert not os.path.exists(tmp_path / "d")
