"""pack_counters / unpack_counters with depth thresholds per tile, on hand-built results (no GPU): the vector is
[6 state counts][5 sums][3 x n_bins bins][hist raw n][hist qc n][territory T][callable T][raw_sum T][qc_sum T]
[raw_ge K x T][qc_ge K x T], threshold-major, the histograms, tiles and thresholds only when they are on; unpack_counters
takes K from res.tile_thresholds."""
import copy

import numpy as np
import pytest

from decodingustools_b200.callable_loci import INTERVAL_DTYPE, ContigDeviceResult
from decodingustools_b200.sharding import TILE_FIELDS, pack_counters, unpack_counters

GE_FIELDS = ("tile_raw_ge", "tile_qc_ge")


def _result(n_bins, n_hist, n_tiles, k, seed):
    rng = np.random.default_rng(seed)
    arr = lambda *shape: rng.integers(0, 2**40, shape).astype(np.uint64)     # noqa: E731
    r = ContigDeviceResult(rng.integers(0, 2**40, 6).astype(np.uint64), *(int(x) for x in rng.integers(0, 2**40, 5)),
                           np.zeros(0, INTERVAL_DTYPE), rng.integers(0, 2**31, (3, n_bins)).astype(np.uint32), 1000, 0, 5000,
                           depth_hist_raw=arr(n_hist) if n_hist else None, depth_hist_qc=arr(n_hist) if n_hist else None)
    if n_tiles:
        r.tile_len = 1000
        for f in TILE_FIELDS:
            setattr(r, f, arr(n_tiles))
    if k:
        r.tile_thresholds = np.cumsum(rng.integers(1, 50, k)).astype(np.uint32)
        r.tile_raw_ge, r.tile_qc_ge = arr(k, n_tiles), arr(k, n_tiles)
    return r


def _blank(res):
    b = copy.deepcopy(res)
    b.state_counts[:] = 0; b.bins[:] = 0
    for f in ("n_covered_bases", "summed_coverage", "summed_baseq", "summed_mapq", "quality_bases"):
        setattr(b, f, 0)
    for f in ("depth_hist_raw", "depth_hist_qc") + TILE_FIELDS + GE_FIELDS:
        if getattr(b, f) is not None:
            setattr(b, f, np.zeros_like(getattr(b, f)))
    return b


@pytest.mark.parametrize("n_bins,n_hist,n_tiles,k", [(7, 0, 1, 1), (7, 0, 3, 8), (1, 1001, 250, 4), (0, 65536, 2, 2), (5, 0, 40, 8)])
def test_thresholds_follow_the_tiles_threshold_major_and_round_trip(n_bins, n_hist, n_tiles, k):
    r = _result(n_bins, n_hist, n_tiles, k, n_tiles + k)
    v = pack_counters(r).view(np.uint64)
    t0 = 11 + 3 * n_bins + 2 * n_hist
    g0 = t0 + 4 * n_tiles
    assert v.shape == (g0 + 2 * k * n_tiles,)
    for i, f in enumerate(TILE_FIELDS):
        assert v[t0 + i * n_tiles:t0 + (i + 1) * n_tiles].tolist() == getattr(r, f).tolist()
    for j in range(k):                                                   # raw_ge[j] then, after all of them, qc_ge[j]
        assert v[g0 + j * n_tiles:g0 + (j + 1) * n_tiles].tolist() == r.tile_raw_ge[j].tolist()
        assert v[g0 + (k + j) * n_tiles:g0 + (k + j + 1) * n_tiles].tolist() == r.tile_qc_ge[j].tolist()
    back = unpack_counters(v.view(np.int64), _blank(r))
    for f in TILE_FIELDS + GE_FIELDS + (("depth_hist_raw", "depth_hist_qc") if n_hist else ()):
        assert np.array_equal(getattr(back, f), getattr(r, f)), f
    assert back.tile_raw_ge.shape == (k, n_tiles) and back.tile_qc_ge.shape == (k, n_tiles)
    assert np.array_equal(back.bins, r.bins) and back.state_counts.tolist() == r.state_counts.tolist()
    assert back.tile_thresholds.tolist() == r.tile_thresholds.tolist()


@pytest.mark.parametrize("n_hist", [0, 300])
def test_without_thresholds_the_vector_is_unchanged(n_hist):
    r = _result(7, n_hist, 20, 0, 5)
    v = pack_counters(r).view(np.uint64)
    assert v.shape == (11 + 21 + 2 * n_hist + 4 * 20,)
    back = unpack_counters(v.view(np.int64), _blank(r))
    assert all(getattr(back, f) is None for f in GE_FIELDS + ("tile_thresholds",))
    assert np.array_equal(back.tile_qc_sum, r.tile_qc_sum)


def test_summed_vectors_sum_the_threshold_counts():
    a, b = _result(5, 17, 40, 3, 10), _result(5, 17, 40, 3, 11)
    b.tile_thresholds = a.tile_thresholds.copy()                         # shards of one contig count at the same thresholds
    s = unpack_counters((pack_counters(a).view(np.uint64) + pack_counters(b).view(np.uint64)).view(np.int64), _blank(a))
    for f in TILE_FIELDS + GE_FIELDS:
        assert np.array_equal(getattr(s, f), getattr(a, f) + getattr(b, f)), f
    assert np.array_equal(s.depth_hist_raw, a.depth_hist_raw + b.depth_hist_raw) and np.array_equal(s.bins, a.bins + b.bins)
