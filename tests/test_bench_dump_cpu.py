"""bench.py --dump-outputs, host side: the file set, its dtypes, the size budget and the seeded row sample."""
import os

import numpy as np

import bench


def _step_outputs(n, m, k, seed=3):
    r = np.random.default_rng(seed)
    return {"idx": r.integers(0, m, (n, k), dtype=np.int32), "dist": r.random((n, k)),
            "counts": r.integers(0, k + 1, (n, k), dtype=np.uint8), "weights": r.random((n, k)), "scores": r.random(m)}


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f), allow_pickle=False) for f in sorted(os.listdir(d))}


def test_small_output_is_written_whole_and_exact(tmp_path):
    out = _step_outputs(700, 900, 7)
    assert bench.dump_outputs(str(tmp_path), out) == (700, 700)
    got = _load(str(tmp_path))
    assert sorted(got) == ["counts", "dist", "idx", "rows", "scores", "weights"]
    assert all(v.dtype in (np.float32, np.float64) for v in got.values())
    assert np.array_equal(got["rows"], np.arange(700))
    for name, v in out.items():
        assert np.array_equal(got[name], v), name


def test_large_output_is_a_seeded_row_sample_within_the_budget(tmp_path):
    out = _step_outputs(20_000, 5_000, 30)
    budget = 2_000_000
    a, b = str(tmp_path / "a"), str(tmp_path / "b")
    keep, n = bench.dump_outputs(a, out, budget)
    assert n == 20_000 and 0 < keep < n
    assert bench.dump_outputs(b, out, budget) == (keep, n)
    assert sum(os.path.getsize(os.path.join(a, f)) for f in os.listdir(a)) <= budget
    got, again = _load(a), _load(b)
    for name in got:
        assert np.array_equal(got[name], again[name]), name            # same arguments, same files
    rows = got["rows"].astype(np.int64)
    assert len(rows) == keep and (np.diff(rows) > 0).all()
    for name in ("idx", "dist", "counts", "weights"):
        assert np.array_equal(got[name], out[name][rows]), name
    assert np.array_equal(got["scores"], out["scores"])


def test_default_budget_is_64_mb():
    assert bench.DUMP_BYTES <= 64 * 10 ** 6
