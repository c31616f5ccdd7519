"""bench.py --dump-outputs (CPU-only): the files hold the match list exactly, stay within the size budget, and a list too
long for it is sampled the same way on every run."""
import os

import numpy as np

import bench
from frizbee_b200 import MATCH_DTYPE


def _matches(n, seed):
    rng = np.random.default_rng(seed)
    m = np.zeros(n, dtype=MATCH_DTYPE)
    m["index"] = rng.permutation(n) + 70_000_000   # beyond 2**24: a float32 index would round
    m["score"] = rng.integers(0, 65536, n)
    m["exact"] = rng.integers(0, 2, n)
    return m


def _load(d):
    return {f[len("matches_"):-len(".npy")]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def test_short_list_is_written_whole_and_exact(tmp_path):
    m = _matches(1000, 1)
    bench.dump_outputs(str(tmp_path), m)
    got = _load(tmp_path)
    assert sorted(got) == ["count", "exact", "index", "score"]
    assert got["index"].dtype == np.float64 and got["score"].dtype == np.float32 and got["exact"].dtype == np.float32
    assert got["count"].tolist() == [1000]
    for f in ("index", "score", "exact"):
        assert np.array_equal(got[f], m[f].astype(np.float64)), f


def test_long_list_is_a_fixed_sample_within_the_budget(tmp_path):
    n = bench.DUMP_BYTES // 16 + 1
    m = _matches(n, 2)
    a, b = tmp_path / "a", tmp_path / "b"
    bench.dump_outputs(str(a), m)
    bench.dump_outputs(str(b), m)
    assert sum(os.path.getsize(a / f) for f in os.listdir(a)) <= bench.DUMP_BYTES
    got = _load(a)
    assert got["count"].tolist() == [n]
    pos = got["position"].astype(np.int64)
    assert len(pos) < n and np.all(np.diff(pos) > 0) and pos[-1] < n
    for f in ("index", "score", "exact"):
        assert np.array_equal(got[f], m[f][pos].astype(np.float64)), f
    again = _load(b)
    assert all(np.array_equal(got[k], again[k]) for k in got)
