"""QC depth runs (clb_set_qc_depth_runs / CallableLociContext.set_qc_depth_runs): the QC depth of every position (the depth
the states are called on, behind quality_bases) as runs of equal depth, segmented in phase C of all three pileup kernels
beside the raw depth runs and compacted like them, against the run-length encoding of the oracle's per-base QC depth.

Every kernel case runs in a default context (fast kernel for ordinary windows) and in a CLB_FORCE_GENERAL=1 context (every
window through the general kernel), with the QC runs off, on alone, and on together with the raw runs: intervals, state
counts, sums, bins and the raw runs must not change, and each run stream must be what it is alone."""
import os
import shutil
import stat
import subprocess
import threading

import numpy as np
import pytest

from decodingustools_b200 import synth
from decodingustools_b200._lib import ClbError
from decodingustools_b200.callable_loci import (RUN_DTYPE, CallableLociContext, admit_reads, compact_reads,
                                                depth_run_ends, stitch_depth_runs)
from decodingustools_b200.options import CallableOptions, CalledState
from tests import bamio
from tests import handover_inputs as H
from tests.helpers import assert_parity, run_oracle

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "decodingustools_b200", "decodingus-tools-b200")
GOLDEN = os.path.join(ROOT, "tests", "golden")
SUMS = ("n_covered_bases", "summed_coverage", "summed_baseq", "summed_mapq", "quality_bases")
# misc words the library copies back: 9, 11 with raw runs, 13 with QC runs (the QC cursor and count follow the raw ones)
MISC_WORDS = {(False, False): 9, (True, False): 11, (False, True): 13, (True, True): 13}


@pytest.fixture(scope="module")
def contexts():
    """contexts(opt) -> (default context, forced-general context), created once per options (CLB_FORCE_GENERAL is read by
    clb_create)."""
    made = {}

    def pair(opt):
        key = (opt.min_depth, opt.max_depth, opt.min_mapping_quality, opt.min_base_quality)
        if key not in made:
            mp = pytest.MonkeyPatch()
            try:
                mp.delenv("CLB_FORCE_GENERAL", raising=False)
                default = CallableLociContext(opt)
                mp.setenv("CLB_FORCE_GENERAL", "1")
                forced = CallableLociContext(opt)
            finally:
                mp.undo()
            made[key] = (default, forced)
        return made[key]

    yield pair
    for default, forced in made.values():
        default.close()
        forced.close()


def rle(depth, lo=0):
    """Runs of equal depth of the per-base depths `depth` (positions lo, lo + 1, ...)."""
    depth = np.asarray(depth, np.int64)
    out = np.zeros(0, RUN_DTYPE)
    if depth.size:
        s = np.flatnonzero(np.r_[True, depth[1:] != depth[:-1]])
        out = np.zeros(s.size, RUN_DTYPE)
        out["start"] = s + lo
        out["depth"] = depth[s]
    return out


def _same_runs(what, got, want):
    assert got is not None, what
    if not np.array_equal(got, want):
        n = min(len(got), len(want))
        bad = np.flatnonzero(got[:n] != want[:n])
        i = int(bad[0]) if bad.size else n
        pytest.fail(f"{what}: {len(got)} runs, want {len(want)}; first difference at run {i}: "
                    f"got {got[i] if i < len(got) else None}, want {want[i] if i < len(want) else None}")


def check_qc_runs(what, res, want, opt):
    """The QC runs equal `want`, and satisfy on their own what every result must: they tile the region, adjacent runs differ,
    the depths add up to quality_bases, and every position's QC depth agrees with its BED state."""
    got = res.qc_depth_runs
    _same_runs(what, got, want)
    starts = got["start"].astype(np.int64)
    ends = depth_run_ends(got, res.region_end)
    lens = ends - starts
    assert (starts[0] if len(got) else res.region_start) == res.region_start, what
    assert (lens > 0).all(), what
    assert (np.diff(got["depth"].astype(np.int64)) != 0).all(), f"{what}: adjacent runs of equal QC depth"
    assert int((lens * got["depth"]).sum()) == res.quality_bases, what
    # the runs against the intervals, position by position
    iv = res.intervals
    assert int(iv["start"][0]) == res.region_start and int(iv["end"][-1]) == res.region_end, what
    assert (iv["start"][1:] == iv["end"][:-1]).all(), what
    qc = np.repeat(got["depth"].astype(np.int64), lens)
    st = np.repeat(iv["state"], (iv["end"] - iv["start"]).astype(np.int64))
    assert (qc[st == CalledState.NO_COVERAGE] == 0).all(), f"{what}: QC depth in NO_COVERAGE"
    assert (qc[st == CalledState.LOW_COVERAGE] < opt.min_depth).all(), f"{what}: QC depth in LOW_COVERAGE"
    call = qc[st == CalledState.CALLABLE]
    assert (call >= opt.min_depth).all() and (opt.max_depth <= 0 or (call <= opt.max_depth).all()), f"{what}: QC depth in CALLABLE"
    if opt.max_depth > 0:
        assert (qc[st == CalledState.EXCESSIVE_COVERAGE] > opt.max_depth).all(), f"{what}: QC depth in EXCESSIVE_COVERAGE"


def same_result(what, on, off):
    assert np.array_equal(on.intervals, off.intervals), what
    assert on.state_counts.tolist() == off.state_counts.tolist(), what
    assert all(getattr(on, k) == getattr(off, k) for k in SUMS), what
    assert np.array_equal(on.bins, off.bins), what


def configure(ctx, raw=False, qc=False, hist=0, tiles=0, thresholds=()):
    ctx.set_depth_runs(raw)
    ctx.set_qc_depth_runs(qc)
    ctx.set_depth_histogram(hist)
    ctx.set_depth_tiles(tiles)
    ctx.set_depth_thresholds(thresholds)


def run_case(pair, contig, opt, hist=0, tiles=0, thresholds=()):
    """Both contexts: assert_parity with no runs, QC runs alone, raw runs alone and both (with the optional counts of the
    last three as given); identical results, QC runs equal to the oracle's, raw runs equal with and without QC runs."""
    name, tid, length, ref, reads = contig
    oc = run_oracle([contig], opt, debug=True).contigs[0]
    want, want_raw = rle(oc.qc), rle(oc.raw)
    extra = 8 * (2 * hist + (4 + 2 * len(thresholds)) * (-(-length // tiles) if tiles else 0))
    for ctx in pair:
        configure(ctx)
        _, off = assert_parity([contig], opt, ctx)
        assert off[0].qc_depth_runs is None and off[0].depth_runs is None
        configure(ctx, qc=True, hist=hist, tiles=tiles, thresholds=thresholds)
        _, qc = assert_parity([contig], opt, ctx)
        same_result(name, qc[0], off[0])
        assert qc[0].depth_runs is None
        check_qc_runs(name, qc[0], want, opt)
        misc = 4 * (MISC_WORDS[(False, True)] - MISC_WORDS[(False, False)])
        assert qc[0].d2h_bytes == off[0].d2h_bytes + misc + 8 * len(want) + extra
        configure(ctx, raw=True, hist=hist, tiles=tiles, thresholds=thresholds)
        _, raw = assert_parity([contig], opt, ctx)
        _same_runs(f"{name} raw", raw[0].depth_runs, want_raw)
        configure(ctx, raw=True, qc=True, hist=hist, tiles=tiles, thresholds=thresholds)
        _, both = assert_parity([contig], opt, ctx)
        same_result(name, both[0], off[0])
        check_qc_runs(f"{name} with raw runs", both[0], want, opt)
        _same_runs(f"{name} raw with QC runs", both[0].depth_runs, raw[0].depth_runs)
        misc = 4 * (MISC_WORDS[(True, True)] - MISC_WORDS[(True, False)])
        assert both[0].d2h_bytes == raw[0].d2h_bytes + misc + 8 * len(want)
        for k in ("depth_hist_raw", "depth_hist_qc", "tile_territory", "tile_callable", "tile_raw_sum", "tile_qc_sum", "tile_raw_ge",
                  "tile_qc_ge"):
            a, b = getattr(both[0], k), getattr(raw[0], k)
            assert (a is None and b is None) or np.array_equal(a, b), (name, k)
        configure(ctx)
    return oc, want


def qc_steps_contig(length=3 * H.WREAL, seed=21):
    """One read at every position, all with a 100-base reference span, so the raw depth is flat (100) away from the ends
    while the QC depth steps: deletions under the pile, reads below min_mapping_quality, low base qualities, qualities
    shorter than the query and 0xFF qualities.  Plus piles the other way round: MAPQ-0 reads and all-low-quality reads
    that step the raw depth where the QC depth stays."""
    rng = np.random.default_rng(seed)
    pos, cigars, mapq, quals = [], [], [], []
    shapes = ["100M", "40M5D55M", "30M2I70M", "10S100M", "60M1D39M"]
    for p in range(length - 100):
        c = shapes[p % len(shapes)]
        ql = H.query_len(c)
        kind = p % 11
        if kind == 3:
            q = np.full(ql, 0xFF, np.uint8)                               # missing qualities
        elif kind == 7:
            q = rng.integers(0, 256, ql // 2).astype(np.uint8)           # shorter than the query
        else:
            q = rng.choice(np.array([2, 12, 23, 37, 130, 200, 255], np.uint8), size=ql)
        pos.append(p); cigars.append(c); mapq.append(5 if p % 13 == 4 else 60); quals.append(q)
    for s in (H.WREAL // 2, H.WREAL + 700, 2 * H.WREAL + 300):
        pos += [s] * 40; cigars += ["100M"] * 40; mapq += [0] * 40; quals += [np.full(100, 37, np.uint8)] * 40
        pos += [s + 250] * 40; cigars += ["100M"] * 40; mapq += [60] * 40; quals += [np.full(100, 2, np.uint8)] * 40
    order = np.argsort(np.array(pos), kind="stable")
    return H.reference(length, seed), H.columns([pos[i] for i in order], [cigars[i] for i in order], np.array([mapq[i] for i in order], np.uint8),
                                                [quals[i] for i in order])


def seam_steps_contig(kind):
    """The 8-window hand-over layout with one 100M read of quality 30 at every position (raw = QC = 100), and at every
    window seam s a step of one depth only.  kind "raw": 50 MAPQ-0 reads start at s, the raw depth steps and the QC depth
    does not (the QC run across the seam continues).  kind "qc": 50 reads of quality 2 end at s and 50 reads of quality 30
    start at it, the QC depth steps and the raw depth does not."""
    seams = [w * H.WREAL for w in range(1, H.SEAM_WINDOWS)]
    pos = list(range(0, H.SEAM_LEN - 100))
    mapq = [60] * len(pos)
    quals = [np.full(100, 30, np.uint8)] * len(pos)
    for s in seams:
        if kind == "raw":
            pos += [s] * 50; mapq += [0] * 50; quals += [np.full(100, 30, np.uint8)] * 50
        else:
            pos += [s - 100] * 50; mapq += [60] * 50; quals += [np.full(100, 2, np.uint8)] * 50
            pos += [s] * 50; mapq += [60] * 50; quals += [np.full(100, 30, np.uint8)] * 50
    order = np.argsort(np.array(pos), kind="stable")
    return H.reference(H.SEAM_LEN, 5), H.columns([pos[i] for i in order], ["100M"] * len(pos), np.array([mapq[i] for i in order], np.uint8),
                                                 [quals[i] for i in order])


def mapq0_contig(length=6 * H.WREAL, seed=9):
    """~40x of MAPQ-0 and MAPQ-60 reads, with MAPQ-0 piles on window seams: the QC depth only sees the MAPQ-60 reads."""
    rng = np.random.default_rng(seed)
    starts = list(np.sort(rng.integers(0, length - 100, int(40 * length / 100))))
    mapq = list(rng.choice([0, 0, 60], size=len(starts)))
    for s in range(H.WREAL, length - 100, H.WREAL):
        starts += [s - 50] * 100 + [s - 50] * 100
        mapq += [0] * 100 + [60] * 100
    order = np.argsort(np.array(starts), kind="stable")
    pos = [int(starts[i]) for i in order]
    mq = np.array([mapq[i] for i in order], np.uint8)
    return H.reference(length, seed, [(3000, 3100)]), H.columns(pos, ["100M"] * len(pos), mq, H.rotating_quals([100] * len(pos), step=7))


# ------------------------------------------------------------------------------------------------ kernel coverage
def test_synthetic_30x_contig(contexts):
    c = synth.synth_short("chr9", 300_000, seed=77)
    _, want = run_case(contexts(CallableOptions()), (c.name, 0, c.length, c.ref, c.reads), CallableOptions())
    assert len(want) > 10_000


@pytest.mark.parametrize("min_bq", [20, 129])
def test_qc_depth_steps_under_a_flat_raw_depth(contexts, min_bq):
    """min_base_quality 129: the BQ_HI instantiations (byte compare of qualities >= 128)."""
    opt = CallableOptions(min_base_quality=min_bq)
    ref, reads = qc_steps_contig()
    oc, want = run_case(contexts(opt), ("chrF", 0, len(ref), ref, reads), opt)
    raw, qc = oc.raw.astype(np.int64), oc.qc.astype(np.int64)
    flat = np.flatnonzero(raw[1:] == raw[:-1]) + 1
    assert (qc[flat] != qc[flat - 1]).sum() > 500                         # QC steps where raw does not
    raw_steps = np.flatnonzero(raw[1:] != raw[:-1]) + 1
    assert (qc[raw_steps] == qc[raw_steps - 1]).sum() > 0                 # ... and the converse


@pytest.mark.parametrize("kind", ["raw", "qc"])
def test_one_depth_steps_at_every_window_seam(contexts, kind):
    """The soft first run of each fast window is dropped by its own kind's window table: with raw steps only, every QC run
    crosses the seam; with QC steps only, every seam starts a QC run and no raw run."""
    ref, reads = seam_steps_contig(kind)
    oc, want = run_case(contexts(CallableOptions()), ("chrZ", 0, H.SEAM_LEN, ref, reads), CallableOptions())
    seams = np.arange(1, H.SEAM_WINDOWS) * H.WREAL
    raw, qc = oc.raw.astype(np.int64), oc.qc.astype(np.int64)
    if kind == "raw":
        assert (raw[seams] != raw[seams - 1]).all() and (qc[seams] == qc[seams - 1]).all()
        assert not np.isin(seams, want["start"]).any()
    else:
        assert (raw[seams] == raw[seams - 1]).all() and (qc[seams] != qc[seams - 1]).all()
        assert np.isin(seams, want["start"]).all()


@pytest.mark.parametrize("feature", H.SEAM_FEATURES)
def test_hand_over_contig_with_features_at_window_seams(contexts, feature):
    ref, reads = H.seam_contig(feature)
    run_case(contexts(CallableOptions()), ("chrZ", 0, H.SEAM_LEN, ref, reads), CallableOptions())


def test_deep_window(contexts):
    """More than 65535 candidates in one window: k_pileup_classify_deep."""
    opt = CallableOptions(max_depth=100_000, min_base_quality=129)
    reads = H.deep_quality_window()
    run_case(contexts(opt), ("chrD", 0, 3 * H.WREAL, H.reference(3 * H.WREAL, 4), reads), opt)
    assert reads.n > 65535


def deep_pile():
    """70000 reads of 50M at one position of window 1 over 200 reads of 100M: QC depths past 16 bits (WIDE arrays)."""
    pos = sorted([30 * i for i in range(200)] + [H.WREAL + 500] * 70_000)
    cigars = ["50M" if p == H.WREAL + 500 else "100M" for p in pos]
    quals = [np.full(int(c[:-1]), 40, np.uint8) for c in cigars]
    return H.columns(pos, cigars, 60, quals)


def test_deep_pile_past_16_bits(contexts):
    opt = CallableOptions(max_depth=100_000)
    oc, want = run_case(contexts(opt), ("chrP", 0, 3 * H.WREAL, H.reference(3 * H.WREAL, 6), deep_pile()), opt)
    assert int(oc.qc.max()) > 65535 and int(want["depth"].max()) > 65535


def test_long_read_contig(contexts):
    c = synth.synth_long("chr2", 120_000, seed=78, depth=20.0)
    run_case(contexts(CallableOptions()), (c.name, 0, c.length, c.ref, c.reads), CallableOptions())


def test_2000x_pile(contexts):
    opt = CallableOptions(max_depth=4000)
    c = synth.synth_short("chrY", 12_000, seed=4, depth=2000.0)
    oc, _ = run_case(contexts(opt), (c.name, 0, c.length, c.ref, c.reads), opt)
    assert int(oc.qc.max()) > 1000


def test_mapq0_piles(contexts):
    ref, reads = mapq0_contig()
    oc, _ = run_case(contexts(CallableOptions()), ("chrQ", 0, len(ref), ref, reads), CallableOptions())
    assert int(oc.low.max()) > 100


def test_contig_without_reads(contexts):
    opt = CallableOptions()
    for ctx in contexts(opt):
        for raw in (False, True):
            configure(ctx, raw=raw, qc=True)
            ctx.begin_contig(0, "chrE", 5000, H.reference(5000, 3), 5000)
            res = ctx.finish_contig()
            assert res.qc_depth_runs.tolist() == [(0, 0)]
            check_qc_runs("empty", res, rle(np.zeros(5000)), opt)
        configure(ctx)


@pytest.mark.parametrize("length", [1000, 3 * H.WREAL])
def test_short_and_window_multiple_contigs(contexts, length):
    c = synth.synth_short("chrS", length, seed=length)
    run_case(contexts(CallableOptions()), (c.name, 0, c.length, c.ref, c.reads), CallableOptions())


def test_everything_on(contexts):
    """Feature set 31: histograms, tiles, thresholds, raw runs and QC runs."""
    c = synth.synth_short("chr3", 200_000, seed=83)
    run_case(contexts(CallableOptions()), (c.name, 0, c.length, c.ref, c.reads), CallableOptions(), hist=1001, tiles=1000,
             thresholds=(1, 10, 20, 30))


# ------------------------------------------------------------------------------------------------ region shards
def test_region_shards_stitch_to_the_whole_contig(contexts):
    """Shards that start at a QC step, inside a QC run and at window multiples: each shard's QC runs are the oracle's over
    the shard, and stitched they are the whole contig's."""
    opt = CallableOptions()
    ref, reads = H.seam_contig("depth_step")
    length = H.SEAM_LEN
    oc = run_oracle([("chrZ", 0, length, ref, reads)], opt, debug=True).contigs[0]
    qc = oc.qc.astype(np.int64)
    at_step = 2 * H.WREAL + 100 + int(np.flatnonzero(qc[2 * H.WREAL + 100:] != qc[2 * H.WREAL + 99:-1])[0])
    inside = 4 * H.WREAL + 100 + int(np.flatnonzero(qc[4 * H.WREAL + 100:] == qc[4 * H.WREAL + 99:-1])[0])
    assert qc[at_step] != qc[at_step - 1] and qc[inside] == qc[inside - 1]
    adm = compact_reads(reads, admit_reads(reads, opt.pileup_max_depth, 0))
    span, end = adm.max_ref_span(), adm.end()
    cuts = [0, H.WREAL, at_step, inside, 5 * H.WREAL, length]
    for ctx in contexts(opt):
        for raw in (False, True):
            configure(ctx, raw=raw, qc=True)
            parts = []
            for a, b in zip(cuts[:-1], cuts[1:]):
                ctx.begin_contig(0, "chrZ", length, ref, length, region=(a, b), max_ref_span=span)
                ctx.push_reads(adm.select((adm.pos < b) & (end > a - 1)))
                res = ctx.finish_contig()
                check_qc_runs(f"shard [{a},{b})", res, rle(qc[a:b], a), opt)
                parts.append(res.qc_depth_runs)
            assert np.array_equal(stitch_depth_runs(parts), rle(qc))
        configure(ctx)


# ------------------------------------------------------------------------------------------------ repeated and re-run work
def test_reruns_debug_runs_and_refresh_return_the_same_runs(contexts):
    opt = CallableOptions()
    c = synth.synth_short("chr4", 100_000, seed=79)
    contig = (c.name, 0, c.length, c.ref, c.reads)
    oc = run_oracle([contig], opt, debug=True).contigs[0]
    want = rle(oc.qc)
    for ctx in contexts(opt):
        configure(ctx, qc=True)
        _, results = assert_parity([contig], opt, ctx)
        _, r1 = ctx.rerun_resident(fetch=True, copy_intervals=True)
        _, r2 = ctx.rerun_resident(fetch=True, copy_intervals=True)
        ctx.debug_per_base(c.length)
        r3 = ctx.refresh_counters()
        for what, r in (("finish", results[0]), ("rerun 1", r1), ("rerun 2", r2), ("refresh after debug", r3)):
            check_qc_runs(what, r, want, opt)
        configure(ctx)


def test_record_capacity_rerun_keeps_the_runs(contexts):
    """REF_N at every other position: more state-run starts than the first record buffer holds, so clb_finish_contig grows
    it and re-runs the contig; the QC run cursor must start from zero again."""
    opt = CallableOptions()
    length = 120_000
    ref = bytearray(H.reference(length, 12))
    ref[1:100_000:2] = b"N" * len(range(1, 100_000, 2))
    c = synth.synth_short("chrR", length, seed=80, depth=12.0)
    run_case(contexts(opt), ("chrR", 0, length, bytes(ref), c.reads), opt)


# ------------------------------------------------------------------------------------------------ switching and errors
def test_switching_raw_and_qc_runs_between_contigs(contexts):
    opt = CallableOptions()
    a = synth.synth_short("chr5", 60_000, seed=81)
    b = synth.synth_short("chr6", 30_000, seed=84)
    ca, cb = (a.name, 0, a.length, a.ref, a.reads), (b.name, 1, b.length, b.ref, b.reads)
    oa, ob = run_oracle([ca], opt, debug=True).contigs[0], run_oracle([cb], opt, debug=True).contigs[0]
    steps = [((True, True), ca, oa), ((False, True), cb, ob), ((True, False), ca, oa), ((False, False), cb, ob),
             ((False, True), ca, oa), ((True, True), cb, ob), ((False, False), ca, oa), ((True, False), cb, ob),
             ((True, True), ca, oa)]
    for ctx in contexts(opt):
        for (raw, qc), contig, oc in steps:
            configure(ctx, raw=raw, qc=qc)
            _, res = assert_parity([contig], opt, ctx)
            _, rr = ctx.rerun_resident(fetch=True, copy_intervals=True)
            for r in (res[0], rr):
                if qc:
                    check_qc_runs(contig[0], r, rle(oc.qc), opt)
                else:
                    assert r.qc_depth_runs is None
                if raw:
                    _same_runs(f"{contig[0]} raw", r.depth_runs, rle(oc.raw))
                else:
                    assert r.depth_runs is None
        configure(ctx)


def test_set_qc_depth_runs_while_a_contig_is_open(contexts):
    opt = CallableOptions()
    ctx = contexts(opt)[0]
    c = synth.synth_short("chr7", 20_000, seed=85)
    configure(ctx)
    ctx.begin_contig(0, c.name, c.length, c.ref, c.length)
    with pytest.raises(ClbError) as e:
        ctx.set_qc_depth_runs(True)
    assert e.value.code == -1
    ctx.push_reads(compact_reads(c.reads, admit_reads(c.reads, opt.pileup_max_depth, 0)))
    assert ctx.finish_contig().qc_depth_runs is None


# ------------------------------------------------------------------------------------------------ coverage command
def expected_bedgraph(ocs, kind="qc"):
    lines = []
    for oc in ocs:
        runs = rle(getattr(oc, kind))
        for r, e in zip(runs, depth_run_ends(runs, oc.length)):
            lines.append(f"{oc.name}\t{r['start']}\t{e}\t{r['depth']}\n")
    return "".join(lines)


def _outputs(d):
    return {p: (d / p).read_bytes() for p in sorted(os.listdir(d)) if p.endswith((".bed", ".json", ".html", ".svg"))}


def _cli(cwd, args):
    return subprocess.run([CLI, "coverage", *args], cwd=cwd, capture_output=True, text=True, timeout=600)


def _genome(tmp_path):
    cs = [synth.synth_short("chr1", 120_000, seed=41), synth.synth_short("chr2", 60_000, seed=42),
          synth.synth_short("chrM", 16_569, seed=43, depth=300.0)]
    contigs = [(c.name, tid, c.length, c.ref, c.reads) for tid, c in enumerate(cs)]
    bam = str(tmp_path / "in.bam"); fa = str(tmp_path / "ref.fa")
    bamio.write_bam(bam, [(n, l, r) for n, _, l, _, r in contigs])
    bamio.write_fasta(fa, [(n, ref) for n, _, _, ref, _ in contigs])
    return contigs, bam, fa


def test_cli_qc_bedgraph_of_a_small_genome_alone_and_with_the_raw_bedgraph(tmp_path):
    contigs, bam, fa = _genome(tmp_path)
    for d in ("off", "raw", "qc", "both"):
        (tmp_path / d).mkdir()
    off = _cli(tmp_path / "off", [bam, "-r", fa, "-o", "out.bed"])
    raw = _cli(tmp_path / "raw", [bam, "-r", fa, "-o", "out.bed", "--depth-bedgraph", "depth.bedgraph"])
    qc = _cli(tmp_path / "qc", [bam, "-r", fa, "-o", "out.bed", "--qc-depth-bedgraph", "qc.bedgraph"])
    both = _cli(tmp_path / "both", [bam, "-r", fa, "-o", "out.bed", "--depth-bedgraph", "depth.bedgraph", "--qc-depth-bedgraph", "qc.bedgraph"])
    for p in (off, raw, qc, both):
        assert p.returncode == 0, p.stderr[-2000:]
    ref_outputs = _outputs(tmp_path / "off")
    assert len(ref_outputs) >= 5
    for d in ("raw", "qc", "both"):
        assert _outputs(tmp_path / d) == ref_outputs, d
    ocs = run_oracle(contigs, CallableOptions(), debug=True).contigs
    want = expected_bedgraph(ocs)
    assert (tmp_path / "qc" / "qc.bedgraph").read_text() == want
    assert (tmp_path / "both" / "qc.bedgraph").read_text() == want
    assert (tmp_path / "both" / "depth.bedgraph").read_bytes() == (tmp_path / "raw" / "depth.bedgraph").read_bytes()
    assert not (tmp_path / "raw" / "qc.bedgraph").exists()


def test_cli_qc_bedgraph_of_the_deep_golden_case(tmp_path):
    """mini_config4_deep_cap500 with the QC bedGraph on: the golden outputs stay byte-identical."""
    from tests.golden_cases import cases
    name = "mini_config4_deep_cap500"
    for f in ("in.bam", "in.bam.bai", "ref.fa", "ref.fa.fai"):
        shutil.copy(os.path.join(GOLDEN, name, f), tmp_path / f)
    p = _cli(tmp_path, ["in.bam", "-r", "ref.fa", "-o", "callable_regions.bed", "--qc-depth-bedgraph", "q.bedgraph"])
    assert p.returncode == 0, p.stderr
    assert (tmp_path / "callable_regions.bed").read_bytes() == open(os.path.join(GOLDEN, name, "expected.callable_regions.bed"), "rb").read()
    assert (tmp_path / "summary.json").read_text() == open(os.path.join(GOLDEN, name, "expected.summary.json")).read()
    _, contigs, opt = next(c for c in cases() if c[0] == name)
    ocs = run_oracle([(n, tid, l, ref, r) for tid, (n, l, ref, r) in enumerate(contigs)], opt, debug=True).contigs
    assert (tmp_path / "q.bedgraph").read_text() == expected_bedgraph(ocs)


def test_cli_qc_bedgraph_to_a_fifo_and_to_an_unwritable_path(tmp_path):
    contigs, bam, fa = _genome(tmp_path)
    fifo = tmp_path / "qc.fifo"
    os.mkfifo(fifo)
    got = []
    reader = threading.Thread(target=lambda: got.append(open(fifo, "rb").read()))
    reader.start()
    p = _cli(tmp_path, [bam, "-r", fa, "-o", "out.bed", "--qc-depth-bedgraph", str(fifo)])
    reader.join(timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    assert stat.S_ISFIFO(os.stat(fifo).st_mode)
    ocs = run_oracle(contigs, CallableOptions(), debug=True).contigs
    assert got and got[0].decode() == expected_bedgraph(ocs)
    (tmp_path / "q.bedgraph").mkdir()
    p = _cli(tmp_path, [bam, "-r", fa, "-o", "out.bed", "--qc-depth-bedgraph", str(tmp_path / "q.bedgraph")])
    assert p.returncode == 1, p.stderr[-2000:]
    assert p.stderr.splitlines()[-1] == f"Error: cannot write {tmp_path / 'q.bedgraph'}", p.stderr[-2000:]
