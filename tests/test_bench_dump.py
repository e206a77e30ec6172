"""bench.py --dump-outputs: the arrays are written as float64 .npy, stay under the size cap, keep small arrays whole and
sample large ones at the same indices from run to run (so two builds can be compared output for output)."""
import os

import numpy as np

import bench


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_outputs_under_the_cap(tmp_path):
    big = np.arange(400_000, dtype=np.float32)  # 3.2 MB as float64
    arrays = {"step_result": [1.5, -2.0, 0, 3e-4], "counts": np.linspace(0, 1, 1000), "params": big}
    limit = 2 << 20
    for sub in ("a", "b"):
        bench.dump_outputs(str(tmp_path / sub), arrays, limit=limit)
    a, b = _load(str(tmp_path / "a")), _load(str(tmp_path / "b"))
    assert set(a) == {"step_result", "counts", "params"}
    assert all(v.dtype == np.float64 for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= limit
    np.testing.assert_array_equal(a["step_result"], [1.5, -2.0, 0, 3e-4])
    np.testing.assert_array_equal(a["counts"], np.linspace(0, 1, 1000))
    assert 0 < a["params"].size < big.size and np.all(np.diff(a["params"]) > 0)  # a sorted subset of the elements
    assert np.isin(a["params"], big).all()
    for k in a:
        np.testing.assert_array_equal(a[k], b[k])


def test_dump_outputs_whole_when_small(tmp_path):
    x = np.random.default_rng(3).standard_normal((20, 30))
    bench.dump_outputs(str(tmp_path), {"x": x})
    np.testing.assert_array_equal(np.load(str(tmp_path / "x.npy")), x.ravel())
