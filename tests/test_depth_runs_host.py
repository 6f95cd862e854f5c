"""Host half of the depth runs (no GPU): the bedGraph writer (clb_bedgraph_writer_*) against plain Python formatting, in
memory, through pwrite, through a FIFO and into /dev/full, its refusal of runs that do not tile the contig, and the shard
stitching and run ends of the Python layer."""
import os
import threading

import numpy as np
import pytest

from decodingustools_b200 import _lib
from decodingustools_b200.callable_loci import RUN_DTYPE, BedGraphWriter, depth_run_ends, stitch_depth_runs


def runs_of(starts, depths):
    r = np.zeros(len(starts), RUN_DTYPE)
    r["start"] = starts
    r["depth"] = depths
    return r


def python_bedgraph(contigs):
    out = []
    for name, length, runs in contigs:
        for r, e in zip(runs.tolist(), depth_run_ends(runs, length).tolist()):
            out.append(f"{name}\t{r[0]}\t{e}\t{r[1]}\n")
    return "".join(out).encode()


def random_contigs(seed):
    """Several contigs: one with more than 65536 runs (the threaded formatter), one reaching 2^32 - 1 with depths up to
    2^32 - 1, zero-length contigs before, between and after, and a one-run contig."""
    rng = np.random.default_rng(seed)
    n = 150_000
    lens = rng.integers(1, 3000, size=n)
    big = runs_of(np.cumsum(lens) - lens, rng.integers(0, 300, size=n))
    huge_len = 2**32 - 1
    starts = np.r_[0, np.sort(rng.choice(np.arange(1, 2**32 - 1, dtype=np.int64), size=999, replace=False))]
    depths = rng.integers(0, 2**32, size=1000, dtype=np.int64)
    depths[-1] = 2**32 - 1
    huge = runs_of(starts, depths)
    return [("chrE0", 0, np.zeros(0, RUN_DTYPE)), ("chrBig", int(lens.sum()), big), ("chrE1", 0, np.zeros(0, RUN_DTYPE)),
            ("chrHuge", huge_len, huge), ("chrOne", 5, runs_of([0], [0])), ("chrE2", 0, np.zeros(0, RUN_DTYPE))]


@pytest.mark.parametrize("seed", [1, 2])
def test_bedgraph_in_memory_and_through_pwrite_equals_python_formatting(tmp_path, seed):
    contigs = random_contigs(seed)
    want = python_bedgraph(contigs)
    mem = BedGraphWriter(None)
    for name, length, runs in contigs:
        mem.add_contig(name, length, runs)
    assert mem.text() == want
    mem.close()
    path = str(tmp_path / "d.bedgraph")
    f = BedGraphWriter(path)
    for name, length, runs in contigs:
        f.add_contig(name, length, runs)
    f.close()
    assert open(path, "rb").read() == want


def test_bedgraph_through_a_fifo():
    """A pipe cannot seek: the threaded parts are written in order."""
    import tempfile
    contigs = random_contigs(3)
    want = python_bedgraph(contigs)
    with tempfile.TemporaryDirectory() as d:
        fifo = os.path.join(d, "d.fifo")
        os.mkfifo(fifo)
        got = []
        reader = threading.Thread(target=lambda: got.append(open(fifo, "rb").read()))
        reader.start()
        try:
            w = BedGraphWriter(fifo)
            try:
                for name, length, runs in contigs:
                    w.add_contig(name, length, runs)
            finally:
                w.close()
        finally:
            reader.join()
    assert got == [want]


def test_bedgraph_into_dev_full_is_an_io_error():
    contigs = random_contigs(4)
    full = BedGraphWriter("/dev/full")
    with pytest.raises(_lib.ClbError) as e:
        full.add_contig(*contigs[1])                                   # threaded: written in add_contig
    assert e.value.code == _lib.CLB_E_IO and "cannot write /dev/full" in str(e.value)
    with pytest.raises(_lib.ClbError) as e:
        full.close()
    assert e.value.code == _lib.CLB_E_IO
    full = BedGraphWriter("/dev/full")
    full.add_contig("s", 7, runs_of([0, 3], [1, 2]))                  # buffered: the failure shows at close
    with pytest.raises(_lib.ClbError) as e:
        full.close()
    assert e.value.code == _lib.CLB_E_IO


def test_bedgraph_refuses_runs_that_do_not_tile_the_contig():
    bad = [
        (10, runs_of([1, 5], [1, 2])),                                 # does not start at 0
        (10, runs_of([0, 5, 5], [1, 2, 3])),                           # starts do not ascend strictly
        (10, runs_of([0, 6, 4], [1, 2, 3])),
        (10, runs_of([0, 10], [1, 2])),                                # a run starts at the contig end
        (10, np.zeros(0, RUN_DTYPE)),                                  # nothing for a non-empty contig
        (0, runs_of([0], [0])),                                        # a run in an empty contig
    ]
    w = BedGraphWriter(None)
    for length, runs in bad:
        with pytest.raises(_lib.ClbError) as e:
            w.add_contig("c", length, runs)
        assert e.value.code == -1
    assert w.text() == b""
    w.add_contig("c", 10, runs_of([0, 9], [4, 4]))                     # tiling is all it asks for
    assert w.text() == b"c\t0\t9\t4\nc\t9\t10\t4\n"
    w.close()


def test_depth_run_ends():
    r = runs_of([100, 105, 230], [3, 0, 7])
    assert depth_run_ends(r, 400).tolist() == [105, 230, 400]
    assert depth_run_ends(np.zeros(0, RUN_DTYPE), 400).tolist() == []


def test_stitch_depth_runs_drops_a_shard_first_run_of_equal_depth_only():
    a = runs_of([0, 10], [1, 2])
    b = runs_of([20, 25], [2, 3])                                      # continues a's last run
    c = runs_of([40], [5])                                             # does not
    d = np.zeros(0, RUN_DTYPE)                                         # an empty shard changes nothing
    e = runs_of([60, 61], [5, 0])                                      # continues c's run across the empty shard
    got = stitch_depth_runs([a, b, d, c, e])
    assert got.tolist() == [(0, 1), (10, 2), (25, 3), (40, 5), (61, 0)]
    assert stitch_depth_runs([]).dtype == RUN_DTYPE and len(stitch_depth_runs([d])) == 0


def test_stitched_shards_of_a_random_depth_track_are_its_runs():
    rng = np.random.default_rng(5)
    depth = np.repeat(rng.integers(0, 4, size=3000), rng.integers(1, 9, size=3000))
    def rle(x, lo):
        s = np.flatnonzero(np.r_[True, x[1:] != x[:-1]])
        return runs_of(s + lo, x[s])
    cuts = [0] + sorted(rng.choice(np.arange(1, depth.size), size=12, replace=False).tolist()) + [depth.size]
    shards = [rle(depth[a:b], a) for a, b in zip(cuts[:-1], cuts[1:])]
    assert np.array_equal(stitch_depth_runs(shards), rle(depth, 0))
