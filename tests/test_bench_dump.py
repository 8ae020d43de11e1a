"""bench.py --dump-outputs: the lists of the last timed step, written so that two builds compare list for list."""
import os
import sys

import numpy as np
import pytest

import bench

NAMES = ("scores", "doc_ids", "query_rows")


def _lists(nq, k):
    rng = np.random.default_rng(5)
    scores = -np.sort(-rng.random((nq, k), dtype=np.float32), axis=1)
    ids = rng.integers(0, 21_015_324, size=(nq, k), dtype=np.int32)       # beyond float32's exact integers
    return scores, ids


def _load(d):
    return [np.load(os.path.join(d, f"{n}.npy")) for n in NAMES]


def test_small_batch_is_dumped_whole(tmp_path):
    s, d = _lists(300, 10)
    assert bench.dump_outputs(str(tmp_path / "out"), s, d) == 300
    got_s, got_d, rows = _load(tmp_path / "out")
    assert (got_s.dtype, got_d.dtype, rows.dtype) == (np.float32, np.float64, np.float64)
    assert np.array_equal(got_s, s) and np.array_equal(got_d.astype(np.int32), d)
    assert np.array_equal(rows, np.arange(300))


def test_large_batch_is_a_fixed_sample_under_the_size_cap(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 1_000_000)
    s, d = _lists(20_000, 10)
    n = bench.dump_outputs(str(tmp_path / "a"), s, d)
    assert 0 < n < 20_000
    assert sum(os.path.getsize(tmp_path / "a" / f"{x}.npy") for x in NAMES) <= 1_000_000
    got_s, got_d, rows = _load(tmp_path / "a")
    r = rows.astype(np.int64)
    assert len(r) == n and np.all(np.diff(r) > 0) and r[-1] < 20_000
    assert np.array_equal(got_s, s[r]) and np.array_equal(got_d.astype(np.int32), d[r])
    bench.dump_outputs(str(tmp_path / "b"), s, d)
    assert np.array_equal(_load(tmp_path / "b")[2], rows)                     # the same rows on every run


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--warmup", "-1"]])
def test_step_counts_are_checked(monkeypatch, argv):
    monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
    with pytest.raises(SystemExit) as e:
        bench.main()
    assert e.value.code == 2
