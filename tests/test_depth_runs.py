"""Depth runs (clb_set_depth_runs / CallableLociContext.set_depth_runs): the raw depth of every position as runs of equal
depth, segmented in phase C of all three pileup kernels and compacted like the intervals, against the run-length encoding of
the oracle's per-base raw depth.

Every kernel case runs in a default context (fast kernel for ordinary windows) and in a CLB_FORCE_GENERAL=1 context (every
window through the general kernel), with the runs off and on: intervals, state counts, sums and bins must not change."""
import os
import shutil
import stat
import subprocess
import threading

import numpy as np
import pytest

from decodingustools_b200 import synth
from decodingustools_b200._lib import ClbError
from decodingustools_b200.callable_loci import (RUN_DTYPE, CallableLociContext, admit_reads, compact_reads, depth_run_ends,
                                                stitch_depth_runs)
from decodingustools_b200.options import CallableOptions
from tests import bamio
from tests import handover_inputs as H
from tests.helpers import assert_parity, run_oracle

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "decodingustools_b200", "decodingus-tools-b200")
GOLDEN = os.path.join(ROOT, "tests", "golden")
SUMS = ("n_covered_bases", "summed_coverage", "summed_baseq", "summed_mapq", "quality_bases")


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


def rle(raw, lo=0):
    """Runs of equal depth of the per-base raw depths raw (positions lo, lo + 1, ...)."""
    raw = np.asarray(raw, np.int64)
    out = np.zeros(0, RUN_DTYPE)
    if raw.size:
        s = np.flatnonzero(np.r_[True, raw[1:] != raw[:-1]])
        out = np.zeros(s.size, RUN_DTYPE)
        out["start"] = s + lo
        out["depth"] = raw[s]
    return out


def check_runs(what, res, want):
    got = res.depth_runs
    assert got is not None, what
    if not np.array_equal(got, want):
        n = min(len(got), len(want))
        bad = np.flatnonzero(got[:n] != want[:n])
        i = int(bad[0]) if bad.size else n
        pytest.fail(f"{what}: {len(got)} runs, want {len(want)}; first difference at run {i}: "
                    f"got {got[i] if i < len(got) else None}, want {want[i] if i < len(want) else None}")
    # what every result must satisfy on its own
    starts = got["start"].astype(np.int64)
    ends = depth_run_ends(got, res.region_end)
    lens = ends - starts
    assert (starts[0] if len(got) else res.region_start) == res.region_start, what
    assert (lens > 0).all(), what
    assert (np.diff(got["depth"].astype(np.int64)) != 0).all(), f"{what}: adjacent runs of equal depth"
    assert int((lens * got["depth"]).sum()) == res.summed_coverage, what
    assert int(lens[got["depth"] > 0].sum()) == res.n_covered_bases, what


def same_result(what, on, off):
    assert np.array_equal(on.intervals, off.intervals), what
    assert on.state_counts.tolist() == off.state_counts.tolist(), what
    assert all(getattr(on, k) == getattr(off, k) for k in SUMS), what
    assert np.array_equal(on.bins, off.bins), what


def run_case(pair, contig, opt, hist=0, tiles=0):
    """Both contexts: assert_parity with the runs off and on (BED, counts, sums, bins, export), identical results, and runs
    equal to the oracle's."""
    name, tid, length, ref, reads = contig
    oc = run_oracle([contig], opt, debug=True).contigs[0]
    want = rle(oc.raw)
    for ctx in pair:
        ctx.set_depth_runs(False)
        _, off = assert_parity([contig], opt, ctx)
        assert off[0].depth_runs is None
        ctx.set_depth_histogram(hist)
        ctx.set_depth_tiles(tiles)
        ctx.set_depth_runs(True)
        _, on = assert_parity([contig], opt, ctx)
        same_result(name, on[0], off[0])
        check_runs(name, on[0], want)
        assert on[0].d2h_bytes == off[0].d2h_bytes + 8 * (1 + len(want)) + 8 * (2 * hist + 4 * len(on[0].tile_territory if tiles else []))
        ctx.set_depth_runs(False)
        ctx.set_depth_histogram(0)
        ctx.set_depth_tiles(0)
    return oc, want


def flat_seam_contig():
    """The 8-window hand-over layout (300-read piles in windows 2, 3 and 5: fast, fast, general, general, fast, general,
    fast, fast) with one 100M read starting at every position: the raw depth is 100 on both sides of every seam, so every
    window-soft first run must be dropped."""
    pos = list(range(0, H.SEAM_LEN - 100))
    for w in H.SEAM_PILES:
        pos += [w * H.WREAL + 1000] * 300
    pos.sort()
    return H.reference(H.SEAM_LEN, 5), H.columns(pos, ["100M"] * len(pos), 60, H.rotating_quals([100] * len(pos), step=19))


def mapq0_contig(length=6 * H.WREAL, seed=9):
    """~40x of MAPQ-0 and MAPQ-60 reads, with 200-read MAPQ-0 piles on window seams: the low-MAPQ half of the packed depth
    word is non-zero almost everywhere and changes where the raw depth does not."""
    rng = np.random.default_rng(seed)
    starts = list(np.sort(rng.integers(0, length - 100, int(40 * length / 100))))
    mapq = list(rng.choice([0, 0, 60], size=len(starts)))
    for s in range(H.WREAL, length - 100, H.WREAL):
        starts += [s - 50] * 100 + [s - 50] * 100
        mapq += [0] * 100 + [60] * 100                                  # same raw depth step, different low-MAPQ mix
    order = np.argsort(np.array(starts), kind="stable")
    pos = [int(starts[i]) for i in order]
    mq = np.array([mapq[i] for i in order], np.uint8)
    return H.reference(length, seed, [(3000, 3100)]), H.columns(pos, ["100M"] * len(pos), mq, H.rotating_quals([100] * len(pos), step=7))


# ------------------------------------------------------------------------------------------------ kernel coverage
def test_synthetic_30x_contig(contexts):
    c = synth.synth_short("chr9", 300_000, seed=77)
    _, want = run_case(contexts(CallableOptions()), (c.name, 0, c.length, c.ref, c.reads), CallableOptions())
    assert len(want) > 10_000


@pytest.mark.parametrize("feature", H.SEAM_FEATURES)
def test_hand_over_contig_with_features_at_window_seams(contexts, feature):
    ref, reads = H.seam_contig(feature)
    run_case(contexts(CallableOptions()), ("chrZ", 0, H.SEAM_LEN, ref, reads), CallableOptions())


def test_equal_depth_on_both_sides_of_every_seam(contexts):
    ref, reads = flat_seam_contig()
    oc, want = run_case(contexts(CallableOptions()), ("chrZ", 0, H.SEAM_LEN, ref, reads), CallableOptions())
    seams = np.arange(1, H.SEAM_WINDOWS) * H.WREAL
    assert (oc.raw[seams] == oc.raw[seams - 1]).all() and not np.isin(seams, want["start"]).any()


def test_deep_window(contexts):
    """More than 65535 candidates in one window: k_pileup_classify_deep (WIDE: 32-bit raw depth, > 65535 here)."""
    opt = CallableOptions(max_depth=100_000, min_base_quality=129)
    reads = H.deep_quality_window()
    run_case(contexts(opt), ("chrD", 0, 3 * H.WREAL, H.reference(3 * H.WREAL, 4), reads), opt)
    assert reads.n > 65535


def deep_pile():
    """70000 reads of 50M at one position of window 1, over 200 reads of 100M spread across windows 0 to 2: more than 65535
    candidates (k_pileup_classify_deep) and raw depths past 16 bits, which only its 32-bit (WIDE) depth arrays hold."""
    pos = sorted([30 * i for i in range(200)] + [H.WREAL + 500] * 70_000)
    cigars = ["50M" if p == H.WREAL + 500 else "100M" for p in pos]
    return H.columns(pos, cigars, 60, H.rotating_quals([int(c[:-1]) for c in cigars], step=11))


def test_deep_pile_past_16_bits(contexts):
    opt = CallableOptions(max_depth=100_000)
    oc, want = run_case(contexts(opt), ("chrP", 0, 3 * H.WREAL, H.reference(3 * H.WREAL, 6), deep_pile()), opt)
    assert int(oc.raw.max()) > 65535 and int(want["depth"].max()) > 65535


def test_long_read_contig(contexts):
    c = synth.synth_long("chr2", 120_000, seed=78, depth=20.0)
    run_case(contexts(CallableOptions()), (c.name, 0, c.length, c.ref, c.reads), CallableOptions())


def test_2000x_pile(contexts):
    opt = CallableOptions(max_depth=4000)
    c = synth.synth_short("chrY", 12_000, seed=4, depth=2000.0)
    oc, _ = run_case(contexts(opt), (c.name, 0, c.length, c.ref, c.reads), opt)
    assert int(oc.raw.max()) > 1000


def test_mapq0_piles(contexts):
    ref, reads = mapq0_contig()
    oc, _ = run_case(contexts(CallableOptions()), ("chrQ", 0, len(ref), ref, reads), CallableOptions())
    assert int(oc.low.max()) > 100


def test_contig_without_reads(contexts):
    opt = CallableOptions()
    for ctx in contexts(opt):
        ctx.set_depth_runs(True)
        ctx.begin_contig(0, "chrE", 5000, H.reference(5000, 3), 5000)
        res = ctx.finish_contig()
        assert res.depth_runs.tolist() == [(0, 0)]
        check_runs("empty", res, rle(np.zeros(5000)))
        ctx.set_depth_runs(False)


@pytest.mark.parametrize("length", [1000, 3 * H.WREAL])
def test_short_and_window_multiple_contigs(contexts, length):
    c = synth.synth_short("chrS", length, seed=length)
    run_case(contexts(CallableOptions()), (c.name, 0, c.length, c.ref, c.reads), CallableOptions())


def test_runs_with_histograms_and_tiles(contexts):
    c = synth.synth_short("chr3", 200_000, seed=83)
    run_case(contexts(CallableOptions()), (c.name, 0, c.length, c.ref, c.reads), CallableOptions(), hist=1001, tiles=1000)


# ------------------------------------------------------------------------------------------------ region shards
@pytest.mark.parametrize("feature", ["depth_step", "continue"])
def test_region_shards_stitch_to_the_whole_contig(contexts, feature):
    """Shards cut at window multiples (their first windows are general, with the halo entry): each shard's runs are the
    oracle's over the shard, and stitched they are the whole contig's."""
    opt = CallableOptions()
    ref, reads = H.seam_contig(feature)
    length = H.SEAM_LEN
    oc = run_oracle([("chrZ", 0, length, ref, reads)], opt, debug=True).contigs[0]
    adm = compact_reads(reads, admit_reads(reads, opt.pileup_max_depth, 0))
    span, end = adm.max_ref_span(), adm.end()
    cuts = [0, 2 * H.WREAL, 4 * H.WREAL, 5 * H.WREAL, length]
    for ctx in contexts(opt):
        ctx.set_depth_runs(True)
        parts = []
        for a, b in zip(cuts[:-1], cuts[1:]):
            ctx.begin_contig(0, "chrZ", length, ref, length, region=(a, b), max_ref_span=span)
            ctx.push_reads(adm.select((adm.pos < b) & (end > a - 1)))
            res = ctx.finish_contig()
            check_runs(f"shard [{a},{b})", res, rle(oc.raw[a:b], a))
            parts.append(res.depth_runs)
        assert np.array_equal(stitch_depth_runs(parts), rle(oc.raw))
        ctx.set_depth_runs(False)


# ------------------------------------------------------------------------------------------------ repeated and re-run work
def test_reruns_debug_runs_and_refresh_return_the_same_runs(contexts):
    opt = CallableOptions()
    c = synth.synth_short("chr4", 100_000, seed=79)
    contig = (c.name, 0, c.length, c.ref, c.reads)
    oc = run_oracle([contig], opt, debug=True).contigs[0]
    want = rle(oc.raw)
    for ctx in contexts(opt):
        ctx.set_depth_runs(True)
        _, results = assert_parity([contig], opt, ctx)
        _, r1 = ctx.rerun_resident(fetch=True)
        _, r2 = ctx.rerun_resident(fetch=True)
        ctx.debug_per_base(c.length)
        r3 = ctx.refresh_counters()
        for what, r in (("finish", results[0]), ("rerun 1", r1), ("rerun 2", r2), ("refresh after debug", r3)):
            check_runs(what, r, want)
        ctx.set_depth_runs(False)


def test_record_capacity_rerun_keeps_the_runs(contexts):
    """REF_N at every other position: more state-run starts than the first record buffer holds, so clb_finish_contig grows
    it and re-runs the contig; the depth-run cursor must start from zero again."""
    opt = CallableOptions()
    length = 120_000
    ref = bytearray(H.reference(length, 12))
    ref[1:100_000:2] = b"N" * len(range(1, 100_000, 2))
    c = synth.synth_short("chrR", length, seed=80, depth=12.0)
    run_case(contexts(opt), ("chrR", 0, length, bytes(ref), c.reads), opt)


# ------------------------------------------------------------------------------------------------ switching and errors
def test_switching_runs_off_and_on_between_contigs(contexts):
    opt = CallableOptions()
    a = synth.synth_short("chr5", 60_000, seed=81)
    b = synth.synth_short("chr6", 30_000, seed=84)
    ca, cb = (a.name, 0, a.length, a.ref, a.reads), (b.name, 1, b.length, b.ref, b.reads)
    wa = rle(run_oracle([ca], opt, debug=True).contigs[0].raw)
    wb = rle(run_oracle([cb], opt, debug=True).contigs[0].raw)
    for ctx in contexts(opt):
        for on, contig, want in ((True, ca, wa), (False, cb, wb), (True, cb, wb), (False, ca, wa), (True, ca, wa)):
            ctx.set_depth_runs(on)
            _, res = assert_parity([contig], opt, ctx)
            if on:
                check_runs(contig[0], res[0], want)
            else:
                assert res[0].depth_runs is None
                _, rr = ctx.rerun_resident(fetch=True)
                assert rr.depth_runs is None
        ctx.set_depth_runs(False)


def test_set_depth_runs_while_a_contig_is_open(contexts):
    opt = CallableOptions()
    ctx = contexts(opt)[0]
    c = synth.synth_short("chr7", 20_000, seed=85)
    ctx.set_depth_runs(False)
    ctx.begin_contig(0, c.name, c.length, c.ref, c.length)
    with pytest.raises(ClbError) as e:
        ctx.set_depth_runs(True)
    assert e.value.code == -1
    ctx.push_reads(compact_reads(c.reads, admit_reads(c.reads, opt.pileup_max_depth, 0)))
    assert ctx.finish_contig().depth_runs is None


# ------------------------------------------------------------------------------------------------ coverage command
def expected_bedgraph(ocs):
    lines = []
    for oc in ocs:
        runs = rle(oc.raw)
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


def test_cli_bedgraph_of_a_small_genome(tmp_path):
    contigs, bam, fa = _genome(tmp_path)
    (tmp_path / "off").mkdir(); (tmp_path / "on").mkdir()
    off = _cli(tmp_path / "off", [bam, "-r", fa, "-o", "out.bed"])
    on = _cli(tmp_path / "on", [bam, "-r", fa, "-o", "out.bed", "--depth-bedgraph", "depth.bedgraph"])
    assert off.returncode == 0 and on.returncode == 0, (off.stderr, on.stderr)
    assert _outputs(tmp_path / "on") == _outputs(tmp_path / "off") and len(_outputs(tmp_path / "off")) >= 5
    ocs = run_oracle(contigs, CallableOptions(), debug=True).contigs
    assert (tmp_path / "on" / "depth.bedgraph").read_text() == expected_bedgraph(ocs)


def test_cli_bedgraph_of_the_deep_golden_case(tmp_path):
    """mini_config4_deep_cap500 with the bedGraph on: the golden outputs stay byte-identical."""
    from tests.golden_cases import cases
    name = "mini_config4_deep_cap500"
    for f in ("in.bam", "in.bam.bai", "ref.fa", "ref.fa.fai"):
        shutil.copy(os.path.join(GOLDEN, name, f), tmp_path / f)
    p = _cli(tmp_path, ["in.bam", "-r", "ref.fa", "-o", "callable_regions.bed", "--depth-bedgraph", "d.bedgraph"])
    assert p.returncode == 0, p.stderr
    assert (tmp_path / "callable_regions.bed").read_bytes() == open(os.path.join(GOLDEN, name, "expected.callable_regions.bed"), "rb").read()
    assert (tmp_path / "summary.json").read_text() == open(os.path.join(GOLDEN, name, "expected.summary.json")).read()
    _, contigs, opt = next(c for c in cases() if c[0] == name)
    ocs = run_oracle([(n, tid, l, ref, r) for tid, (n, l, ref, r) in enumerate(contigs)], opt, debug=True).contigs
    assert (tmp_path / "d.bedgraph").read_text() == expected_bedgraph(ocs)


def test_cli_bedgraph_to_a_fifo_and_to_an_unwritable_path(tmp_path):
    contigs, bam, fa = _genome(tmp_path)
    fifo = tmp_path / "depth.fifo"
    os.mkfifo(fifo)
    got = []
    reader = threading.Thread(target=lambda: got.append(open(fifo, "rb").read()))
    reader.start()
    p = _cli(tmp_path, [bam, "-r", fa, "-o", "out.bed", "--depth-bedgraph", str(fifo)])
    reader.join(timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    assert stat.S_ISFIFO(os.stat(fifo).st_mode)
    ocs = run_oracle(contigs, CallableOptions(), debug=True).contigs
    assert got and got[0].decode() == expected_bedgraph(ocs)
    (tmp_path / "d.bedgraph").mkdir()
    p = _cli(tmp_path, [bam, "-r", fa, "-o", "out.bed", "--depth-bedgraph", str(tmp_path / "d.bedgraph")])
    assert p.returncode == 1, p.stderr[-2000:]
    assert p.stderr.splitlines()[-1] == f"Error: cannot write {tmp_path / 'd.bedgraph'}", p.stderr[-2000:]
