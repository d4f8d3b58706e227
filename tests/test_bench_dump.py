"""bench.py --dump-outputs: the headline's result rows as .npy files that two builds can be compared by (no GPU needed:
the rows are given in the form cg_partial_fetch returns them)."""
import importlib.util
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_dump_writes_result_rows_by_key_as_float(tmp_path):
    bench = _bench()
    sums = np.array([10, -4, 7, 0, 1], np.int64)
    fetch = dict(n=5, keys=np.array([5, 3, 0, 9, 7], np.int64), key_nulls=np.array([0, 0, 1, 0, 0], np.uint8),
                 sum_hi=np.stack([sums >> 63, np.zeros(5, np.int64)], 1), sum_lo=np.stack([sums, np.zeros(5, np.int64)], 1).view(np.uint64),
                 count=np.array([[1, 1], [2, 2], [1, 3], [0, 4], [1, 1]], np.int64))
    bench.dump_c2_result(str(tmp_path), fetch)
    got = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert sorted(got) == ["count_star", "key", "key_is_null", "sum_v"]
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert got["key"].tolist() == [3, 5, 7, 9, 0] and got["key_is_null"].tolist() == [0, 0, 0, 0, 1]   # NULL group last
    assert np.array_equal(got["sum_v"], [-4, 10, 1, np.nan, 7], equal_nan=True)                        # no input: NULL
    assert got["count_star"].tolist() == [2, 1, 1, 4, 3]
