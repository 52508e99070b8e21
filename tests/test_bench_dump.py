"""bench.py --dump-outputs: finite files, at most 64 MB, the same seeded sample of events from every array."""
import os

import numpy as np


def test_dump_keeps_one_seeded_sample_of_events_under_the_cap(tmp_path):
    import torch
    import bench
    n = 20000
    ev = torch.arange(n, dtype=torch.float64)
    arrays = {"rows": ev[:, None].repeat(1, 49), "triggers": ev[:, None, None].repeat(1, 16, 32)}   # 4.5 KB per event
    for d in ("a", "b"):
        bench.dump_outputs(torch, str(tmp_path / d), arrays)
    files = [f"{k}{s}.npy" for k in arrays for s in ("", "_nonfinite")]
    assert sorted(os.listdir(tmp_path / "a")) == sorted(files)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= bench.DUMP_BYTES
    rows, trig = (np.load(tmp_path / "a" / f"{k}.npy") for k in arrays)
    assert rows.dtype == trig.dtype == np.float64
    assert 0 < len(rows) < n and np.all(np.diff(rows[:, 0]) > 0)
    assert np.array_equal(rows[:, 0], trig[:, 0, 0])
    for f in files:
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))
    bench.dump_outputs(torch, str(tmp_path / "small"), {"rows": arrays["rows"][:100]})
    assert np.array_equal(np.load(tmp_path / "small" / "rows.npy"), arrays["rows"][:100].numpy())


def test_dump_writes_non_finite_outputs_as_codes(tmp_path):
    import torch
    import bench
    a = torch.tensor([[1.5, float("nan")], [float("inf"), -float("inf")]], dtype=torch.float32)
    bench.dump_outputs(torch, str(tmp_path), {"t": a})
    vals, code = np.load(tmp_path / "t.npy"), np.load(tmp_path / "t_nonfinite.npy")
    assert vals.dtype == np.float32 and code.dtype == np.float32
    assert np.array_equal(vals, [[1.5, 0.0], [0.0, 0.0]])
    assert np.array_equal(code, [[0, 1], [2, 3]])
