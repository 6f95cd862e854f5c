"""Host half of the C-ABI library on CPU: symbols, admission, BED writer quirks, stitching, report floats.
No compute call touches a GPU here."""
import os
import re
import threading

import numpy as np
import pytest

from decodingustools_b200 import _lib, report
from decodingustools_b200.callable_loci import (INTERVAL_DTYPE, CallableProfiler, ContigProfiler, admit_reads,
                                                bin_geometry, count_unique_reads, stitch_intervals)
from decodingustools_b200.options import CallableOptions
from decodingustools_b200.soa import ReadColumns, n_mask_from_ascii
from oracle import oracle
from tests.test_oracle_vs_naive import random_reads


def states_to_intervals(states: np.ndarray) -> np.ndarray:
    n = states.shape[0]
    if n == 0:
        return np.zeros(0, INTERVAL_DTYPE)
    starts = np.flatnonzero(np.concatenate([[True], states[1:] != states[:-1]]))
    iv = np.zeros(starts.shape[0], INTERVAL_DTYPE)
    iv["start"] = starts; iv["end"] = np.concatenate([starts[1:], [n]]); iv["state"] = states[starts]
    return iv


def test_library_loads_and_exports_every_declared_symbol():
    L = _lib.lib()
    assert L.clb_abi_version() == 2
    hdr = open(os.path.join(os.path.dirname(_lib._HERE), "include", "callable_loci_b200.h")).read()
    declared = set(re.findall(r"\b(clb_[a-z0-9_]+)\s*\(", hdr))
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    for s in declared:
        assert hasattr(L, s), s


def test_device_path_fails_loudly_without_gpu():
    L = _lib.lib()
    if L.clb_device_count() > 0:
        pytest.skip("GPU present")
    from decodingustools_b200.callable_loci import CallableLociContext
    with pytest.raises(_lib.ClbError):
        CallableLociContext(CallableOptions())


@pytest.mark.parametrize("seed", range(30))
def test_admission_matches_oracle(seed):
    rng = np.random.default_rng(300 + seed)
    reads = random_reads(rng, 40, int(rng.integers(0, 120)))
    for maxcnt in (1, 2, 3, 5, 500):
        for tid in (0, 2):
            assert admit_reads(reads, maxcnt, tid).tolist() == oracle.admit(reads, maxcnt, tid).tolist()


@pytest.mark.parametrize("seed", range(12))
def test_parallel_admission_equals_sequential(seed):
    """clb_admit_reads_mt == clb_admit_reads: sparse stretches (decided independently), deep piles (replayed runs),
    runs that touch, zero-span records, placed-unmapped records, several thread counts."""
    rng = np.random.default_rng(900 + seed)
    recs = []
    p = 0
    for blk in range(int(rng.integers(3, 9))):
        deep = rng.random() < 0.5
        n = int(rng.integers(50, 400)) if deep else int(rng.integers(5, 60))
        for _ in range(n):
            p += int(rng.integers(0, 2 if deep else 40))
            kind = rng.random()
            cig = "30M" if kind < 0.7 else ("10M5D15M" if kind < 0.8 else ("12S" if kind < 0.9 else "5M2I20M"))
            flag = 4 if rng.random() < 0.05 else 0
            recs.append((p, flag, 60, cig, 30, f"r{len(recs)}"))
        p += int(rng.integers(0, 200))
    reads = ReadColumns.from_records(recs)
    for maxcnt in (1, 3, 8, 50):
        for tid in (0, 1):
            want = admit_reads(reads, maxcnt, tid)
            assert want.tolist() == oracle.admit(reads, maxcnt, tid).tolist()
            for threads, span in ((1, 0), (3, 0), (8, 35), (0, 1000)):
                st = {}
                got = admit_reads(reads, maxcnt, tid, threads=threads, max_ref_span=span, stats=st)
                assert got.tolist() == want.tolist(), (maxcnt, tid, threads, span)


def test_parallel_admission_sparse_data_replays_nothing():
    from decodingustools_b200 import synth
    c = synth.synth_short("chr22", 400_000, seed=3)
    st = {}
    keep = admit_reads(c.reads, 500, 0, threads=4, stats=st)
    assert st["replayed"] == 0 and keep.tolist() == admit_reads(c.reads, 500, 0).tolist()
    assert np.array_equal(keep, (c.reads.flag & 4) == 0)


def test_admission_rejects_unsorted():
    reads = ReadColumns.from_records([(5, 0, 60, "3M", 30), (2, 0, 60, "3M", 30)])
    with pytest.raises(_lib.ClbError):
        admit_reads(reads, 500, 0)


@pytest.mark.parametrize("seed", range(12))
def test_bed_writer_reproduces_oracle_bytes_and_bins(seed):
    """Feed the writer intervals derived from the oracle's per-base states; BED bytes (incl. duplicated
    boundary lines) and bins (incl. the stale range) must equal the oracle's."""
    rng = np.random.default_rng(900 + seed)
    names = ["chr1", "chr2", "chrM", "chrX", "chrUn"]
    lens = [int(rng.choice([0, 1, 7, 33, 64])) for _ in names]
    if max(l for n, l in zip(names, lens) if n != "chrM") == 0:
        lens[0] = 9
    largest = max(l for n, l in zip(names, lens) if n != "chrM")
    opt = CallableOptions(min_depth=2, max_depth=4)
    o = oracle.OracleRun(opt, largest)
    prof = CallableProfiler(None, largest)
    for tid, (name, length) in enumerate(zip(names, lens)):
        ref = bytes(rng.choice(list(b"ACGTN"), size=length, p=[.2, .2, .2, .2, .2]).tolist())
        reads = random_reads(rng, max(length, 1), int(rng.integers(0, 40))) if length > 2 else ReadColumns.empty()
        oc = o.process_contig(name, tid, length, ref, reads, debug=True)
        iv = states_to_intervals(oc.state)
        stride, nb = bin_geometry(name, length, largest)
        own = np.zeros((3, nb), np.uint32)
        pos = np.arange(length)
        for row, st in enumerate((1, 5, 0)):
            np.add.at(own[row], pos[oc.state == st] // stride, 1)
        got = prof.add_contig(name, length, iv, oc.counts, own, stride)
        assert (got is None) == (oc.bins is None)
        if got is not None:
            assert got.tolist() == oc.bins.tolist()
    assert prof.bed_bytes() == o.bed()


def test_bed_writer_rejects_gappy_intervals():
    prof = CallableProfiler(None, 10)
    iv = np.zeros(2, INTERVAL_DTYPE); iv["start"] = [0, 6]; iv["end"] = [5, 10]; iv["state"] = [1, 2]
    with pytest.raises(_lib.ClbError):
        prof.add_contig("c", 10, iv, [0] * 6, None, 1)


def test_stitch_merges_soft_seams_only():
    a = np.zeros(2, INTERVAL_DTYPE); a["start"] = [0, 4]; a["end"] = [4, 10]; a["state"] = [2, 1]
    b = np.zeros(2, INTERVAL_DTYPE); b["start"] = [10, 12]; b["end"] = [12, 20]; b["state"] = [1, 3]; b["soft_start"] = [1, 0]
    c = np.zeros(1, INTERVAL_DTYPE); c["start"] = [20]; c["end"] = [30]; c["state"] = [5]
    out = stitch_intervals([a, b, c])
    assert out["start"].tolist() == [0, 4, 12, 20] and out["end"].tolist() == [4, 12, 20, 30]
    assert out["state"].tolist() == [2, 1, 3, 5] and out["soft_start"].tolist() == [0, 0, 0, 0]


def test_bin_geometry():
    assert bin_geometry("chrM", 16569, 248956422) == (83, 16569 // 83 + 1)
    assert bin_geometry("chr1", 248956422, 248956422) == (124479, 248956422 // 124479 + 1)


def test_contig_order_matches_oracle():
    names = ["chr10", "chr2", "chrM", "chrX", "chr1", "chrY", "chrUn_x", "2", "10", "MT", "chr1_random", "X", "chr+5", "chr05"]
    for a in names:
        for b in names:
            assert report.compare_contig_names(a, b) == oracle.compare_contig_names(a, b), (a, b)


def test_report_floats_match_oracle_bitwise():
    rng = np.random.default_rng(77)
    opt = CallableOptions(min_depth=2)
    names = ["chr2", "chr1", "chrX", "chrM"]
    o = oracle.OracleRun(opt, 64)
    prof = CallableProfiler(None, 64)
    stats = {}
    for tid, name in enumerate(names):
        length = 64
        ref = bytes(rng.choice(list(b"ACGTN"), size=length).tolist())
        reads = random_reads(rng, length, 60)
        oc = o.process_contig(name, tid, length, ref, reads, debug=True)
        keep = admit_reads(reads, opt.pileup_max_depth, tid)
        cp = ContigProfiler(name, length, oc.n_covered_bases, oc.summed_coverage, oc.summed_baseq, oc.summed_mapq,
                            oc.quality_bases, count_unique_reads(reads, keep, length))
        assert cp.n_reads == oc.n_reads
        stats[tid] = cp
        prof.add_contig(name, length, states_to_intervals(oc.state), oc.counts, None, 1)
    exp = report.build_coverage_export(stats, prof)
    order, fl, sm = o.export()
    assert [c["name"] for c in exp["contigs"]] == [names[i] for i in order]
    for c, f in zip(exp["contigs"], fl):
        assert c["coverage_percent"] == f["coverage_percent"] and c["average_depth"] == f["average_depth"]
        assert c["quality_stats"] == {k: f[k] for k in ("average_mapq", "average_baseq", "q30_percentage")}
    assert exp["summary"]["average_depth"] == sm["average_depth"]
    assert exp["summary"]["callable_percentage"] == sm["callable_percentage"]
    assert exp["quality_metrics"] == {k: sm[k] for k in ("average_mapq", "average_baseq", "q30_percentage")}
    assert exp["total_unique_reads"] == sm["total_unique_reads"]


def test_nmask_packing():
    ref = b"ACNNnACGTN" * 7
    m = n_mask_from_ascii(ref)
    for p, ch in enumerate(ref):
        assert ((int(m[p >> 5]) >> (p & 31)) & 1) == (ch in b"Nn")


def test_bed_writer_large_contig_threads_and_file(tmp_path):
    """More than 65536 runs: the threaded formatter, in memory and through pwrite, against plain Python formatting;
    a small contig afterwards checks the file offset is left at the end (and quirk Q1 across the two).  Then the same through a
    FIFO, and into /dev/full, which must fail with CLB_E_IO."""
    rng = np.random.default_rng(77)
    n = 150_000
    lens = rng.integers(1, 3000, size=n)
    ends = np.cumsum(lens); starts = ends - lens
    st = rng.integers(0, 6, size=n).astype(np.uint8)
    for i in range(1, n):
        if st[i] == st[i - 1]:
            st[i] = (st[i] + 1) % 6
    iv = np.zeros(n, INTERVAL_DTYPE); iv["start"] = starts; iv["end"] = ends; iv["state"] = st
    L = int(ends[-1])
    names = ["REF_N", "CALLABLE", "NO_COVERAGE", "LOW_COVERAGE", "EXCESSIVE_COVERAGE", "POOR_MAPPING_QUALITY"]
    want = "".join(f"chrBig\t{a}\t{b}\t{names[s]}\n" for a, b, s in zip(starts.tolist(), ends.tolist(), st.tolist()))
    last = want.splitlines()[-1] + "\n"
    small = np.zeros(1, INTERVAL_DTYPE); small["end"] = 7; small["state"] = 2
    want_all = (want + last + "s\t0\t7\tNO_COVERAGE\n").encode()
    mem = CallableProfiler(None, L)
    mem.add_contig("chrBig", L, iv, np.zeros(6), None, 0); mem.add_contig("s", 7, small, np.zeros(6), None, 0)
    assert mem.bed_bytes() == want_all
    path = str(tmp_path / "big.bed")
    f = CallableProfiler(path, L)
    f.add_contig("chrBig", L, iv, np.zeros(6), None, 0); f.add_contig("s", 7, small, np.zeros(6), None, 0)
    f.close()
    assert open(path, "rb").read() == want_all
    # a pipe cannot seek: the parts are written in order
    fifo = str(tmp_path / "bed.fifo")
    os.mkfifo(fifo)
    got = []
    reader = threading.Thread(target=lambda: got.append(open(fifo, "rb").read()))
    reader.start()
    try:
        p = CallableProfiler(fifo, L)
        try:
            p.add_contig("chrBig", L, iv, np.zeros(6), None, 0); p.add_contig("s", 7, small, np.zeros(6), None, 0)
        finally:
            p.close()
    finally:
        reader.join()
    assert got == [want_all]
    # a full disk is an error, whether it shows up in add_contig (large contig) or only when the buffer is flushed at close
    full = CallableProfiler("/dev/full", L)
    with pytest.raises(_lib.ClbError) as e:
        full.add_contig("chrBig", L, iv, np.zeros(6), None, 0)
    assert e.value.code == _lib.CLB_E_IO and "cannot write /dev/full" in str(e.value)
    with pytest.raises(_lib.ClbError) as e:
        full.close()
    assert e.value.code == _lib.CLB_E_IO
    full = CallableProfiler("/dev/full", L)
    full.add_contig("s", 7, small, np.zeros(6), None, 0)
    with pytest.raises(_lib.ClbError) as e:
        full.close()
    assert e.value.code == _lib.CLB_E_IO
