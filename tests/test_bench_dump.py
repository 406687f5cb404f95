"""bench.py --dump-outputs: the arrays of one solve as <dir>/<name>.npy in float64, within the size budget (CPU only)."""
import os

import numpy as np

import bench


def _res(B, T=30, D=7):
    rng = np.random.default_rng(3)
    return dict(x=rng.standard_normal((B, T, D)), status=rng.integers(0, 3, B).astype(np.int32),
                total_cost=rng.standard_normal(B), n_qp_solves=rng.integers(1, 40, B).astype(np.int32),
                timing={"total_ms": 1.0})


def _read(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_writes_every_array_as_float64(tmp_path):
    res = _res(16)
    bench.dump_outputs(str(tmp_path), res)
    got = _read(tmp_path)
    assert sorted(got) == ["n_qp_solves", "status", "total_cost", "x"]
    for k, a in got.items():
        assert a.dtype == np.float64
        np.testing.assert_array_equal(a, res[k])


def test_dump_over_budget_writes_a_fixed_sample(tmp_path):
    res = _res(1000)
    budget = 200_000
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), res, budget=budget)
    a, b = _read(tmp_path / "a"), _read(tmp_path / "b")
    assert sum(os.path.getsize(tmp_path / "a" / (k + ".npy")) for k in a) <= budget
    idx = a["trajectory_index"].astype(int)
    assert 0 < len(idx) < 1000 and (np.diff(idx) > 0).all()
    for k in a:
        np.testing.assert_array_equal(a[k], b[k])
        if k != "trajectory_index":
            np.testing.assert_array_equal(a[k], res[k][idx])
