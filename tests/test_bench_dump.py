"""bench.py --dump-outputs on the host: what it writes, in which layout, and that it stays within 64 MiB.  CPU only."""
import numpy as np
import torch

import bench


def test_dump_outputs_fit_in_64_mib():
    assert (bench.D * bench.DUMP_COLS + bench.NCOLS) * 4 <= 64 << 20


def test_dump_outputs_writes_the_seeded_column_sample(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "NCOLS", 1000)
    monkeypatch.setattr(bench, "DUMP_COLS", 64)
    y = torch.randn(1000, bench.D).t()  # D x N column-major, like the timed path's output
    lj = torch.randn(1000)
    bench.dump_outputs(str(tmp_path / "out"), y, lj)
    ys, ljs = np.load(tmp_path / "out" / "y.npy"), np.load(tmp_path / "out" / "logjac.npy")
    cols = np.sort(np.random.default_rng(0).choice(1000, 64, replace=False))
    assert ys.dtype == np.float32 and ys.shape == (bench.D, 64)
    assert np.array_equal(ys, y.numpy()[:, cols])
    assert ljs.dtype == np.float32 and np.array_equal(ljs, lj.numpy())
    assert sorted(p.name for p in (tmp_path / "out").iterdir()) == ["logjac.npy", "y.npy"]
