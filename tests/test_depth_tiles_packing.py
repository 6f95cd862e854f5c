"""pack_counters / unpack_counters with depth tiles, and the tile geometry, on hand-built results (no GPU): the vector is
[6 state counts][5 sums][3 x n_bins bins][hist raw n][hist qc n][territory T][callable T][raw_sum T][qc_sum T], the
histograms and the tiles only when they are on; tile t covers [t * L, min((t + 1) * L, length))."""
import copy

import numpy as np
import pytest

from decodingustools_b200.callable_loci import INTERVAL_DTYPE, ContigDeviceResult, depth_tile_ranges
from decodingustools_b200.sharding import TILE_FIELDS, pack_counters, unpack_counters


def _result(n_bins, n_hist, n_tiles, seed):
    rng = np.random.default_rng(seed)
    arr = lambda n: rng.integers(0, 2**40, n).astype(np.uint64) if n else None     # noqa: E731
    r = ContigDeviceResult(rng.integers(0, 2**40, 6).astype(np.uint64), *(int(x) for x in rng.integers(0, 2**40, 5)),
                           np.zeros(0, INTERVAL_DTYPE), rng.integers(0, 2**31, (3, n_bins)).astype(np.uint32), 1000, 0, 5000,
                           depth_hist_raw=arr(n_hist), depth_hist_qc=arr(n_hist))
    for f in TILE_FIELDS:
        setattr(r, f, arr(n_tiles))
    return r


def _blank(res):
    b = copy.deepcopy(res)
    b.state_counts[:] = 0; b.bins[:] = 0
    for k in ("n_covered_bases", "summed_coverage", "summed_baseq", "summed_mapq", "quality_bases"):
        setattr(b, k, 0)
    for k in ("depth_hist_raw", "depth_hist_qc") + TILE_FIELDS:
        if getattr(b, k) is not None:
            setattr(b, k, np.zeros_like(getattr(b, k)))
    return b


@pytest.mark.parametrize("n_bins,n_hist,n_tiles", [(7, 0, 1), (7, 0, 3), (1, 1001, 250), (0, 65536, 2)])
def test_tiles_follow_the_histograms_and_round_trip(n_bins, n_hist, n_tiles):
    r = _result(n_bins, n_hist, n_tiles, n_tiles)
    v = pack_counters(r).view(np.uint64)
    t0 = 11 + 3 * n_bins + 2 * n_hist
    assert v.shape == (t0 + 4 * n_tiles,)
    for i, f in enumerate(TILE_FIELDS):
        assert v[t0 + i * n_tiles:t0 + (i + 1) * n_tiles].tolist() == getattr(r, f).tolist()
    if n_hist:
        assert v[11 + 3 * n_bins:t0].tolist() == r.depth_hist_raw.tolist() + r.depth_hist_qc.tolist()
    back = unpack_counters(v.view(np.int64), _blank(r))
    for f in TILE_FIELDS + (("depth_hist_raw", "depth_hist_qc") if n_hist else ()):
        assert np.array_equal(getattr(back, f), getattr(r, f)), f
    assert np.array_equal(back.bins, r.bins) and back.state_counts.tolist() == r.state_counts.tolist()


def test_without_tiles_the_vector_is_unchanged():
    r = _result(7, 300, 0, 5)
    v = pack_counters(r).view(np.uint64)
    assert v.shape == (11 + 21 + 600,)
    back = unpack_counters(v.view(np.int64), _blank(r))
    assert all(getattr(back, f) is None for f in TILE_FIELDS)
    assert np.array_equal(back.depth_hist_qc, r.depth_hist_qc)


def test_summed_vectors_sum_the_tiles():
    a, b = _result(5, 17, 40, 10), _result(5, 17, 40, 11)
    s = unpack_counters((pack_counters(a).view(np.uint64) + pack_counters(b).view(np.uint64)).view(np.int64), _blank(a))
    for f in TILE_FIELDS:
        assert np.array_equal(getattr(s, f), getattr(a, f) + getattr(b, f)), f
    assert np.array_equal(s.depth_hist_raw, a.depth_hist_raw + b.depth_hist_raw) and np.array_equal(s.bins, a.bins + b.bins)


@pytest.mark.parametrize("length,tile_len,n", [(1000, 256, 4), (1024, 256, 4), (1025, 256, 5), (1, 256, 1), (0, 256, 0),
                                               (248_956_422, 1000, 248_957), (300_000, 2**31, 1), (2047, 2047, 1), (2048, 2047, 2)])
def test_tile_geometry(length, tile_len, n):
    start, end = depth_tile_ranges(length, tile_len)
    assert len(start) == len(end) == n
    if n:
        assert start[0] == 0 and end[-1] == length and np.all(end[:-1] == start[1:])
        assert np.all(end[:-1] - start[:-1] == tile_len) and 0 < end[-1] - start[-1] <= tile_len    # only the last may be partial
        assert np.array_equal(start, np.arange(n) * tile_len)
