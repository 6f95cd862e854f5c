"""bench.py --dump-outputs on the CPU: the files written for a result built by hand (the GPU run writes the device's)."""
import os
import sys

import numpy as np
import pytest

import bench
from decodingustools_b200.callable_loci import INTERVAL_DTYPE, ContigDeviceResult


def _result(n):
    iv = np.zeros(n, INTERVAL_DTYPE)
    iv["start"] = np.arange(n, dtype=np.uint32) * 97 + 200_000_000; iv["end"] = iv["start"] + 97; iv["state"] = np.arange(n) % 6
    bins = np.arange(3 * 2001, dtype=np.uint32).reshape(3, 2001)
    return ContigDeviceResult(np.arange(1, 7, dtype=np.uint64), 7, 7_226_012_825, 252_910_448_875, 9, 11, iv, bins, 124_479, 0, int(iv["end"][-1]))


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def test_short_interval_lists_are_written_whole(tmp_path):
    r = _result(1000)
    bench.dump_outputs(str(tmp_path), r)
    got = _load(tmp_path)
    assert all(a.dtype == np.float64 for a in got.values())
    assert got["summed_coverage"] == r.summed_coverage and got["summed_baseq"] == r.summed_baseq and got["stride"] == 124_479
    assert np.array_equal(got["state_counts"], r.state_counts) and np.array_equal(got["bins"], r.bins)
    assert got["n_intervals"] == 1000 and np.array_equal(got["interval_row"], np.arange(1000))
    for k in ("start", "end", "state", "soft_start"):
        assert np.array_equal(got["interval_" + k], r.intervals[k])


def test_long_interval_lists_are_sampled_the_same_way_every_time(tmp_path):
    n = 2 * bench.DUMP_INTERVAL_ROWS + 5
    r = _result(n)
    bench.dump_outputs(str(tmp_path / "a"), r)
    bench.dump_outputs(str(tmp_path / "b"), r)
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)
    rows = a["interval_row"].astype(np.int64)
    assert rows.size == bench.DUMP_INTERVAL_ROWS and np.all(np.diff(rows) > 0) and rows[-1] < n and a["n_intervals"] == n
    assert np.array_equal(a["interval_start"], r.intervals["start"][rows]) and np.array_equal(a["interval_state"], r.intervals["state"][rows])
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 64 << 20


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "d"]])
def test_arguments_that_cannot_be_honoured_are_refused(monkeypatch, argv):
    monkeypatch.setattr(sys, "argv", ["bench.py", *argv])
    with pytest.raises(SystemExit):
        bench.parse_args()
