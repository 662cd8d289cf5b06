"""bench.py on the CPU: --dump-outputs writes float32 .npy files, whole while they fit the size budget and otherwise the
same seeded sample of their elements in every run; --steps below 1 is refused."""
import numpy as np
import pytest
import torch

import bench


def test_dump_outputs_whole_arrays(tmp_path):
    a = torch.randn(2, 4, 8, 8, dtype=torch.float64, generator=torch.Generator().manual_seed(0))
    bench.dump_outputs(str(tmp_path / "d"), {"latents": a})
    got = np.load(tmp_path / "d" / "latents.npy")
    assert got.dtype == np.float32 and got.shape == (2, 4, 8, 8) and np.array_equal(got, a.float().numpy())


def test_dump_outputs_sample_beyond_the_budget(tmp_path):
    arrays = {"a": torch.arange(1000, dtype=torch.float32), "b": torch.arange(3000, dtype=torch.float32).reshape(30, 100)}
    for run in ("r0", "r1"):
        bench.dump_outputs(str(tmp_path / run), arrays, budget=1600)  # 400 of the 4000 elements
    for name, n, size in (("a", 100, 1000), ("b", 300, 3000)):  # every array keeps the same share
        got = np.load(tmp_path / "r0" / f"{name}.npy")
        assert got.dtype == np.float32 and got.shape == (n,)
        assert np.all(np.diff(got) > 0) and got[0] >= 0 and got[-1] < size  # distinct elements, in index order
        assert np.array_equal(got, np.load(tmp_path / "r1" / f"{name}.npy"))  # the same elements in every run
    assert sum(f.stat().st_size for f in (tmp_path / "r0").iterdir()) <= 1600 + 2 * 128  # data + one .npy header each


def test_steps_below_one_refused(monkeypatch):
    monkeypatch.setattr("sys.argv", ["bench.py", "--steps", "0"])
    with pytest.raises(SystemExit) as e:
        bench.main()
    assert e.value.code == 2
