"""pack_counters / unpack_counters with and without depth histograms, on hand-built results (no GPU): the vector is
[6 state counts][5 sums][3 x n_bins bins][raw n][qc n], the histograms only when they are on."""
import copy

import numpy as np

from decodingustools_b200.callable_loci import INTERVAL_DTYPE, ContigDeviceResult
from decodingustools_b200.sharding import pack_counters, unpack_counters


def _result(n_bins, n_hist, seed):
    rng = np.random.default_rng(seed)
    hist = (lambda: rng.integers(0, 2**40, n_hist).astype(np.uint64)) if n_hist else (lambda: None)
    return ContigDeviceResult(rng.integers(0, 2**40, 6).astype(np.uint64), *(int(x) for x in rng.integers(0, 2**40, 5)),
                              np.zeros(0, INTERVAL_DTYPE), rng.integers(0, 2**31, (3, n_bins)).astype(np.uint32), 1000, 0, 5000,
                              depth_hist_raw=hist(), depth_hist_qc=hist())


def _blank(res):
    b = copy.deepcopy(res)
    b.state_counts[:] = 0; b.bins[:] = 0
    for k in ("n_covered_bases", "summed_coverage", "summed_baseq", "summed_mapq", "quality_bases"):
        setattr(b, k, 0)
    if b.depth_hist_raw is not None:
        b.depth_hist_raw = np.zeros_like(b.depth_hist_raw); b.depth_hist_qc = np.zeros_like(b.depth_hist_qc)
    return b


def test_without_histograms_the_vector_is_unchanged():
    r = _result(7, 0, 1)
    v = pack_counters(r).view(np.uint64)
    assert v.shape == (11 + 21,)
    assert v[:6].tolist() == r.state_counts.tolist() and v[11:].tolist() == r.bins.ravel().tolist()
    back = unpack_counters(v.view(np.int64), _blank(r))
    assert back.depth_hist_raw is None and back.depth_hist_qc is None
    assert np.array_equal(back.bins, r.bins) and back.summed_mapq == r.summed_mapq


def test_histograms_follow_the_bins_and_round_trip():
    for n_bins, n in ((7, 2), (1, 1001), (0, 65536)):
        r = _result(n_bins, n, n)
        v = pack_counters(r).view(np.uint64)
        assert v.shape == (11 + 3 * n_bins + 2 * n,)
        assert v[11 + 3 * n_bins:11 + 3 * n_bins + n].tolist() == r.depth_hist_raw.tolist()
        assert v[11 + 3 * n_bins + n:].tolist() == r.depth_hist_qc.tolist()
        back = unpack_counters(v.view(np.int64), _blank(r))
        assert np.array_equal(back.depth_hist_raw, r.depth_hist_raw) and np.array_equal(back.depth_hist_qc, r.depth_hist_qc)
        assert np.array_equal(back.bins, r.bins) and back.state_counts.tolist() == r.state_counts.tolist()


def test_summed_vectors_sum_the_histograms():
    a, b = _result(5, 300, 10), _result(5, 300, 11)
    s = unpack_counters((pack_counters(a).view(np.uint64) + pack_counters(b).view(np.uint64)).view(np.int64), _blank(a))
    assert np.array_equal(s.depth_hist_raw, a.depth_hist_raw + b.depth_hist_raw)
    assert np.array_equal(s.depth_hist_qc, a.depth_hist_qc + b.depth_hist_qc)
    assert np.array_equal(s.bins, a.bins + b.bins)
