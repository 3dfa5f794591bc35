"""bench.py --dump-outputs (host side): float64 arrays, one seeded row sample shared by every per-row array, the
whole dump within its byte limit and identical from run to run."""
import os

import numpy as np
import torch


def test_dump_outputs_sample_and_size(tmp_path, monkeypatch):
    import bench
    # a limit of 8000 bytes forces the row sample (m < n) at n = 1000; small gathers also keep torch's host thread
    # pool from starting before tests/test_sharding_gloo.py forks
    monkeypatch.setattr(bench, "DUMP_BYTES", 8000)
    n = 1000
    rng = np.random.default_rng(0)
    W = np.column_stack([np.arange(n, dtype=np.float64), rng.standard_normal(n)])    # column 0: the row's index
    host = {"Vir": rng.standard_normal(n), "W": W}
    per_row = {k: torch.from_numpy(v) for k, v in host.items()}
    values = {"nll": 1.25, "grad": np.arange(3.0)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), values, per_row, n)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["Vir.npy", "W.npy", "grad.npy", "nll.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in names) <= bench.DUMP_BYTES
    out = {f[:-4]: np.load(tmp_path / "a" / f) for f in names}
    assert all(a.dtype == np.float64 for a in out.values())
    assert all(np.array_equal(a, np.load(tmp_path / "b" / (k + ".npy"))) for k, a in out.items())
    assert out["nll"].tolist() == [1.25] and out["grad"].tolist() == [0.0, 1.0, 2.0]
    rows = out["W"][:, 0].astype(np.int64)
    # the sample drawn with seed 0: as many rows as the limit allows, ascending, the same rows for every array
    assert rows.size == 161 and np.all(np.diff(rows) > 0) and 0 <= rows[0] and rows[-1] < n
    assert rows[:8].tolist() == [2, 4, 7, 13, 16, 19, 24, 29] and rows[-3:].tolist() == [989, 990, 995]
    assert np.array_equal(out["W"], W[rows]) and np.array_equal(out["Vir"], host["Vir"][rows])
    bench.dump_outputs(str(tmp_path / "c"), values, {"Vir": per_row["Vir"][:300]}, 300)   # fits: every row
    assert np.array_equal(np.load(tmp_path / "c" / "Vir.npy"), host["Vir"][:300])
