"""Depth histograms (clb_set_depth_histogram / CallableLociContext.set_depth_histogram): the raw- and QC-depth histograms
of a contig or region shard, counted in phase C of all three pileup kernels, against the oracle's per-base depths.

Expected bin d = positions that are not REF_N with depth min(depth, n - 1) == d.  Every kernel case runs in a default
context (fast kernel for ordinary windows) and in a CLB_FORCE_GENERAL=1 context (every window through the general kernel),
at bin counts on both sides of the fast kernel's 256-entry shared table and of the clamp."""
import json
import os
import shutil
import subprocess

import numpy as np
import pytest

from decodingustools_b200 import synth
from decodingustools_b200._lib import ClbError
from decodingustools_b200.callable_loci import CallableLociContext, admit_reads, compact_reads
from decodingustools_b200.options import CallableOptions
from decodingustools_b200.sharding import pack_counters, unpack_counters
from tests import bamio
from tests import handover_inputs as H
from tests.helpers import assert_parity, run_oracle

pytestmark = pytest.mark.gpu

NS = (2, 17, 255, 256, 257, 1001, 65536)
REF_N, NO_COVERAGE = 0, 2
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "decodingustools_b200", "decodingus-tools-b200")
GOLDEN = os.path.join(ROOT, "tests", "golden")


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


def expected(oc, n, lo=0, hi=None):
    """Oracle histograms of positions [lo, hi) from its per-base dump."""
    own = oc.state[lo:hi] != REF_N
    raw = np.bincount(np.minimum(oc.raw[lo:hi][own], n - 1), minlength=n)
    qc = np.bincount(np.minimum(oc.qc[lo:hi][own], n - 1), minlength=n)
    return raw, qc


def _same(what, got, want):
    assert got is not None, what
    got, want = np.asarray(got, np.uint64), np.asarray(want).astype(np.uint64)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, f"{what}: {bad.size} bins differ, first {bad[0]}: got {got[bad[0]]}, want {want[bad[0]]}"


def check_invariants(res, length, n):
    raw, qc = res.depth_hist_raw, res.depth_hist_qc
    own = length - int(res.state_counts[REF_N])
    assert int(raw.sum()) == int(qc.sum()) == own
    assert int(raw[0]) == int(res.state_counts[NO_COVERAGE])
    if res.state_counts[REF_N] == 0 and raw[n - 1] == 0:              # no clamped depth: the sums follow
        d = np.arange(n, dtype=np.uint64)
        assert int((d * raw).sum()) == res.summed_coverage and int((d * qc).sum()) == res.quality_bases


def run_case(pair, contig, opt, ns=NS):
    """Both contexts, every n: assert_parity with the histograms on (BED, counts, sums, bins, export), histograms equal to
    the oracle's, the invariants, and the counter buffer's length."""
    name, tid, length, ref, reads = contig
    oc = run_oracle([contig], opt, debug=True).contigs[0]
    for ctx in pair:
        for n in ns:
            ctx.set_depth_histogram(n)
            _, results = assert_parity([contig], opt, ctx)
            res = results[0]
            raw, qc = expected(oc, n)
            _same(f"raw n={n}", res.depth_hist_raw, raw)
            _same(f"qc n={n}", res.depth_hist_qc, qc)
            check_invariants(res, length, n)
            assert ctx.counters_device()[1] == 12 + 3 * res.bins.shape[1] + 2 * n
        ctx.set_depth_histogram(0)
    return oc


# ------------------------------------------------------------------------------------------------ kernel coverage
def test_synthetic_30x_contig(contexts):
    c = synth.synth_short("chr9", 300_000, seed=77)
    run_case(contexts(CallableOptions()), (c.name, 0, c.length, c.ref, c.reads), CallableOptions())


@pytest.mark.parametrize("n_pile,n_before", [(254, 300), (255, 300)])
def test_piles_at_the_fast_kernels_depth_limit(contexts, n_pile, n_before):
    """254 reads over one position (fast kernel: the deepest entry of its 256-bin table) and 255 (the fast kernel starts the
    window, sees the 255th read and hands it to the general kernel: nothing it counted may remain)."""
    opt = CallableOptions()
    oc = run_case(contexts(opt), ("chrP", 0, H.DEPTH_LEN, H.reference(H.DEPTH_LEN, 1), H.depth_pile(n_pile, n_before)), opt)
    assert int(oc.raw.max()) == n_pile


def test_deep_window(contexts):
    """More than 65535 candidates in one window: k_pileup_classify_deep."""
    opt = CallableOptions(max_depth=100_000, min_base_quality=129)
    run_case(contexts(opt), ("chrD", 0, 3 * H.WREAL, H.reference(3 * H.WREAL, 4), H.deep_quality_window()), opt)


def test_long_read_contig(contexts):
    c = synth.synth_long("chr2", 120_000, seed=78, depth=20.0)
    run_case(contexts(CallableOptions()), (c.name, 0, c.length, c.ref, c.reads), CallableOptions())


@pytest.mark.parametrize("feature", ["continue", "n_through", "gap_ends", "gap_starts"])
def test_mixed_fast_and_general_windows_with_ref_n_and_gaps_at_seams(contexts, feature):
    """The 8-window contig whose kernels run fast, fast, general, general, fast, general, fast, fast, with REF_N runs or
    coverage gaps across every seam."""
    ref, reads = H.seam_contig(feature)
    run_case(contexts(CallableOptions()), ("chrZ", 0, H.SEAM_LEN, ref, reads), CallableOptions())


def test_uncapped_2000x_pile_fills_bins_past_255_and_the_clamp(contexts):
    opt = CallableOptions(max_depth=4000)
    c = synth.synth_short("chrY", 12_000, seed=4, depth=2000.0)
    oc = run_case(contexts(opt), (c.name, 0, c.length, c.ref, c.reads), opt)
    assert int(oc.raw.max()) > 1001                                     # n = 1001 clamps, n = 65536 does not


# ------------------------------------------------------------------------------------------------ region shards
def test_region_shards_sum_to_the_whole_contig(contexts):
    """Shards cut at window multiples (their first windows are general, with the halo entry) sum to the whole-contig
    histograms, and pack_counters / unpack_counters carry them."""
    opt = CallableOptions()
    ref, reads = H.seam_contig("depth_step")                           # the halo positions carry depth
    length = H.SEAM_LEN
    oc = run_oracle([("chrZ", 0, length, ref, reads)], opt, debug=True).contigs[0]
    adm = compact_reads(reads, admit_reads(reads, opt.pileup_max_depth, 0))
    span, end = adm.max_ref_span(), adm.end()
    cuts = [0, 2 * H.WREAL, 4 * H.WREAL, 5 * H.WREAL, length]
    for ctx in contexts(opt):
        for n in (17, 1001):
            ctx.set_depth_histogram(n)
            parts = []
            for a, b in zip(cuts[:-1], cuts[1:]):
                ctx.begin_contig(0, "chrZ", length, ref, length, region=(a, b), max_ref_span=span)
                ctx.push_reads(adm.select((adm.pos < b) & (end > a - 1)))
                res = ctx.finish_contig()
                raw, qc = expected(oc, n, a, b)
                _same(f"shard [{a},{b}) raw", res.depth_hist_raw, raw); _same(f"shard [{a},{b}) qc", res.depth_hist_qc, qc)
                parts.append(res)
            vec = sum(pack_counters(p).view(np.uint64) for p in parts)
            whole = unpack_counters(vec.view(np.int64), parts[0])
            raw, qc = expected(oc, n)
            _same("summed raw", whole.depth_hist_raw, raw); _same("summed qc", whole.depth_hist_qc, qc)
            assert whole.state_counts.tolist() == oc.counts and whole.summed_coverage == oc.summed_coverage
        ctx.set_depth_histogram(0)


# ------------------------------------------------------------------------------------------------ repeated and re-run work
def test_reruns_debug_runs_and_refresh_return_the_same_histograms(contexts):
    opt = CallableOptions()
    c = synth.synth_short("chr4", 100_000, seed=79)
    contig = (c.name, 0, c.length, c.ref, c.reads)
    oc = run_oracle([contig], opt, debug=True).contigs[0]
    for ctx in contexts(opt):
        ctx.set_depth_histogram(1001)
        _, results = assert_parity([contig], opt, ctx)
        first = results[0]
        _, r1 = ctx.rerun_resident(fetch=True)
        _, r2 = ctx.rerun_resident(fetch=True)
        ctx.debug_per_base(c.length)
        r3 = ctx.refresh_counters()
        raw, qc = expected(oc, 1001)
        for what, r in (("finish", first), ("rerun 1", r1), ("rerun 2", r2), ("refresh after debug", r3)):
            _same(f"{what} raw", r.depth_hist_raw, raw); _same(f"{what} qc", r.depth_hist_qc, qc)
        ctx.set_depth_histogram(0)


def test_record_capacity_rerun_keeps_the_histograms(contexts):
    """REF_N at every other position: more run starts than the first record buffer holds, so clb_finish_contig grows it and
    re-runs the contig from reset accumulators."""
    opt = CallableOptions()
    length = 120_000
    ref = bytearray(H.reference(length, 12))
    ref[1:100_000:2] = b"N" * len(range(1, 100_000, 2))
    c = synth.synth_short("chrR", length, seed=80, depth=12.0)
    run_case(contexts(opt), ("chrR", 0, length, bytes(ref), c.reads), opt, ns=(256, 1001))


# ------------------------------------------------------------------------------------------------ switching and errors
def test_turning_histograms_off_between_contigs(contexts):
    opt = CallableOptions()
    c = synth.synth_short("chr5", 60_000, seed=81)
    contig = (c.name, 0, c.length, c.ref, c.reads)
    for ctx in contexts(opt):
        ctx.set_depth_histogram(1001)
        _, on = assert_parity([contig], opt, ctx)
        ctx.set_depth_histogram(0)
        _, off = assert_parity([contig], opt, ctx)
        assert off[0].depth_hist_raw is None and off[0].depth_hist_qc is None
        assert np.array_equal(on[0].intervals, off[0].intervals) and np.array_equal(on[0].bins, off[0].bins)
        assert on[0].state_counts.tolist() == off[0].state_counts.tolist()
        assert ctx.counters_device()[1] == 12 + 3 * off[0].bins.shape[1]
        _, rr = ctx.rerun_resident(fetch=True)
        assert rr.depth_hist_raw is None


def test_invalid_settings_are_refused(contexts):
    opt = CallableOptions()
    ctx = contexts(opt)[0]
    for n in (1, 65537):
        with pytest.raises(ClbError) as e:
            ctx.set_depth_histogram(n)
        assert e.value.code == -1
    c = synth.synth_short("chr6", 20_000, seed=82)
    ctx.begin_contig(0, c.name, c.length, c.ref, c.length)
    with pytest.raises(ClbError) as e:
        ctx.set_depth_histogram(100)
    assert e.value.code == -1
    ctx.push_reads(compact_reads(c.reads, admit_reads(c.reads, opt.pileup_max_depth, 0)))
    assert ctx.finish_contig().depth_hist_raw is None
    ctx.set_depth_histogram(0)


@pytest.mark.parametrize("forced", [False, True])
def test_refused_batch_then_a_good_contig(forced):
    from tests.test_kernel_handover import _refuse
    opt = CallableOptions()
    mp = pytest.MonkeyPatch()
    try:
        if forced:
            mp.setenv("CLB_FORCE_GENERAL", "1")
        else:
            mp.delenv("CLB_FORCE_GENERAL", raising=False)
        ctx = CallableLociContext(opt)
    finally:
        mp.undo()
    try:
        ref, reads = H.seam_contig("continue")
        contig = ("chrZ", 0, H.SEAM_LEN, ref, reads)
        oc = run_oracle([contig], opt, debug=True).contigs[0]
        ctx.set_depth_histogram(257)
        _refuse(ctx, 3 * H.WREAL, "unsorted")
        _, results = assert_parity([contig], opt, ctx)
        raw, qc = expected(oc, 257)
        _same("raw", results[0].depth_hist_raw, raw); _same("qc", results[0].depth_hist_qc, qc)
    finally:
        ctx.close()


# ------------------------------------------------------------------------------------------------ coverage command
def tsv_rows(name, raw, qc):
    nz = np.flatnonzero((np.asarray(raw) != 0) | (np.asarray(qc) != 0))
    last = int(nz[-1]) + 1 if nz.size else 0
    return [f"{name}\t{d}\t{int(raw[d])}\t{int(qc[d])}" for d in range(last)]


def expected_tsv(ocs, n):
    lines = ["#contig\tdepth\traw_bases\tqc_bases"]
    tot_raw, tot_qc = np.zeros(n, np.int64), np.zeros(n, np.int64)
    for oc in ocs:
        raw, qc = expected(oc, n)
        lines += tsv_rows(oc.name, raw, qc)
        tot_raw += raw; tot_qc += qc
    lines += tsv_rows("*", tot_raw, tot_qc)
    return "\n".join(lines) + "\n"


def _outputs(d):
    return {p: (d / p).read_bytes() for p in sorted(os.listdir(d)) if p.endswith((".bed", ".json", ".html", ".svg"))}


def _cli(cwd, args):
    p = subprocess.run([CLI, "coverage", *args], cwd=cwd, capture_output=True, text=True, timeout=600)
    return p


def test_cli_histogram_of_a_small_genome(tmp_path):
    cs = [synth.synth_short("chr1", 120_000, seed=41), synth.synth_short("chr2", 60_000, seed=42),
          synth.synth_short("chrM", 16_569, seed=43, depth=300.0)]
    contigs = [(c.name, tid, c.length, c.ref, c.reads) for tid, c in enumerate(cs)]
    (tmp_path / "off").mkdir(); (tmp_path / "on").mkdir()
    bam = str(tmp_path / "in.bam"); fa = str(tmp_path / "ref.fa")
    bamio.write_bam(bam, [(n, l, r) for n, _, l, _, r in contigs])
    bamio.write_fasta(fa, [(n, ref) for n, _, _, ref, _ in contigs])
    off = _cli(tmp_path / "off", [bam, "-r", fa, "-o", "out.bed"])
    on = _cli(tmp_path / "on", [bam, "-r", fa, "-o", "out.bed", "--depth-histogram", "depth.tsv"])
    assert off.returncode == 0 and on.returncode == 0, (off.stderr, on.stderr)
    assert _outputs(tmp_path / "on") == _outputs(tmp_path / "off") and len(_outputs(tmp_path / "off")) >= 5
    ocs = run_oracle(contigs, CallableOptions(), debug=True).contigs
    assert (tmp_path / "on" / "depth.tsv").read_text() == expected_tsv(ocs, 1001)


@pytest.mark.parametrize("dmax", [100, 5000])
def test_cli_histogram_of_the_deep_golden_case(tmp_path, dmax):
    """mini_config4_deep_cap500 (depth up to ~500 after the cap) with the last row below and above its deepest position."""
    from tests.golden_cases import cases
    name = "mini_config4_deep_cap500"
    for f in ("in.bam", "in.bam.bai", "ref.fa", "ref.fa.fai"):
        shutil.copy(os.path.join(GOLDEN, name, f), tmp_path / f)
    p = _cli(tmp_path, ["in.bam", "-r", "ref.fa", "-o", "callable_regions.bed", "--depth-histogram", "h.tsv",
                        "--depth-histogram-max", str(dmax)])
    assert p.returncode == 0, p.stderr
    assert (tmp_path / "callable_regions.bed").read_bytes() == open(os.path.join(GOLDEN, name, "expected.callable_regions.bed"), "rb").read()
    assert (tmp_path / "summary.json").read_text() == open(os.path.join(GOLDEN, name, "expected.summary.json")).read()
    _, contigs, opt = next(c for c in cases() if c[0] == name)
    ocs = run_oracle([(n, tid, l, ref, r) for tid, (n, l, ref, r) in enumerate(contigs)], opt, debug=True).contigs
    assert (int(ocs[0].raw.max()) > dmax) == (dmax == 100)
    assert (tmp_path / "h.tsv").read_text() == expected_tsv(ocs, dmax + 1)


def test_cli_unwritable_histogram_path(tmp_path):
    c = synth.synth_short("chr1", 30_000, seed=44)
    bam = str(tmp_path / "in.bam"); fa = str(tmp_path / "ref.fa")
    bamio.write_bam(bam, [(c.name, c.length, c.reads)]); bamio.write_fasta(fa, [(c.name, c.ref)])
    (tmp_path / "h.tsv").mkdir()
    for extra in ([], ["--progress"]):
        p = _cli(tmp_path, [bam, "-r", fa, "-o", "out.bed", "--depth-histogram", str(tmp_path / "h.tsv"), *extra])
        assert p.returncode == 1, p.stderr[-2000:]
        last = p.stderr.splitlines()[-1]
        assert last == f"Error: cannot write {tmp_path / 'h.tsv'}", p.stderr[-2000:]
        if extra:
            events = [json.loads(line) for line in p.stderr.splitlines() if line.startswith("{")]
            assert events[0] == {"Started": {"task": "Coverage Analysis"}}
            assert events[-1] == {"Error": {"task": "Coverage Analysis", "error": last[len("Error: "):]}}
