"""Results never depend on which kernel took a window: every case here runs through the oracle, a default context
(k_pileup_fast for ordinary windows, k_pileup_general / k_pileup_classify_deep for the rest) and a context created with
CLB_FORCE_GENERAL=1 (every window through the general kernel), and all three must agree per base and in every output.
The inputs (tests/handover_inputs.py) sit on both sides of each rule that hands a window from one kernel to the other,
and every case also asserts which kernel the default context used."""
import numpy as np
import pytest

from decodingustools_b200 import _lib, synth
from decodingustools_b200._lib import ClbError
from decodingustools_b200.callable_loci import CallableLociContext, admit_reads, compact_reads, stitch_intervals
from decodingustools_b200.options import CallableOptions
from tests import handover_inputs as H
from tests.helpers import assert_parity, run_oracle
from tests.test_host_half import states_to_intervals

pytestmark = pytest.mark.gpu

U32_MAX = 2**32 - 1
_SUMS = ("n_covered_bases", "summed_coverage", "summed_baseq", "summed_mapq", "quality_bases")


def _options_key(opt):
    return (opt.min_depth, opt.max_depth, opt.min_mapping_quality, opt.min_base_quality, opt.min_depth_for_low_mapq,
            opt.max_low_mapq, float(opt.max_low_mapq_fraction).hex())          # hex: -0.0 and 0.0 are different contexts


@pytest.fixture(scope="module")
def contexts():
    """contexts(opt) -> (default context, forced-general context) for these options, created once per module.
    clb_create reads CLB_FORCE_GENERAL once, so the variable only has to be set while the second one is created."""
    made = {}

    def pair(opt=None):
        opt = opt or CallableOptions()
        key = _options_key(opt)
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

    pair()
    yield pair
    for default, forced in made.values():
        default.close()
        forced.close()


def _same(what, got, want):
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, f"{what}: {bad.size} positions differ, first at {bad[0]}: got {got[bad[0]]}, want {want[bad[0]]}"


def _admitted(reads, opt, tid=0):
    return compact_reads(reads, admit_reads(reads, opt.pileup_max_depth, tid))


def _check_context(ctx, contig, opt, oc):
    """One context against the oracle: BED bytes, counts, sums and bins (assert_parity), the intervals, the per-base
    raw / qc / low / state of the debug instantiations, and the result of those instantiations against the production one."""
    name, tid, length, ref, reads = contig
    _, results = assert_parity([contig], opt, ctx)
    res = results[0]
    want = states_to_intervals(oc.state)
    for f in ("start", "end", "state"):
        _same(f"interval {f}", res.intervals[f], want[f])
    raw, qc, low, st = ctx.debug_per_base(length)
    _same("raw", raw, oc.raw); _same("qc", qc, oc.qc); _same("low", low, oc.low); _same("state", st, oc.state)
    dbg = ctx.refresh_counters()
    assert np.array_equal(dbg.intervals, res.intervals) and np.array_equal(dbg.state_counts, res.state_counts)
    assert np.array_equal(dbg.bins, res.bins)
    for k in _SUMS:
        assert getattr(dbg, k) == getattr(res, k), k
    return res


def run_three(pair, contig, opt):
    """The contig through the oracle (debug), the default context and the forced-general context; both contexts must
    match the oracle bit for bit.  The forced context must have taken every window through the general kernel, and the
    default context exactly the windows the host model of the routing predicts.  Returns the default run's
    general_windows."""
    name, tid, length, ref, reads = contig
    oc = run_oracle([contig], opt, debug=True).contigs[0]
    default, forced = pair
    n_w = -(-length // H.WREAL)
    gw_forced = _check_context(forced, contig, opt, oc).general_windows
    assert gw_forced == n_w, (gw_forced, n_w)
    gw = _check_context(default, contig, opt, oc).general_windows
    plans = H.plan_windows(_admitted(reads, opt, tid), length, min_mapq=opt.min_mapping_quality)
    assert gw == H.general_count(plans), (gw, [(p.w, p.reason) for p in plans if p.reason])
    return gw


def test_window_size_matches_the_library():
    assert int(_lib.lib().clb_window_positions()) == H.WREAL


# ------------------------------------------------------------------------------------------------ 1. depth proof
@pytest.mark.parametrize("n_pile,n_before,path", [(254, 300, "fast"), (254, 254, "fast"), (255, 254, "general"), (255, 300, "general")])
def test_depth_proof_piles(contexts, n_pile, n_before, path):
    """A pile of exactly 254 reads over one position stays on the fast kernel; 255 go to the general kernel.  With
    n_before = 254 the sampled proof of k_window_ranges catches the pile up front; with n_before = 300 no sample
    (r_lo + 254 k, r_lo = 0 here) lands on the pile's 255th read, so only the fast kernel's per-read check sees it and
    the window is handed over in flight."""
    reads = H.depth_pile(n_pile, n_before)
    gw = run_three(contexts(), ("chrP", 0, H.DEPTH_LEN, H.reference(H.DEPTH_LEN, 1), reads), CallableOptions())
    assert gw == (0 if path == "fast" else 1)


# ------------------------------------------------------------------------------------------------ 2. quality bytes
@pytest.mark.parametrize("copies", [1, 4])
@pytest.mark.parametrize("min_bq", H.QUAL_THRESHOLDS)
def test_quality_bytes_at_every_threshold(contexts, min_bq, copies):
    """Every quality byte 0..255 against thresholds on both sides of 128 (bytes_ge / bytes_lt with BQ_HI), segments of 1..16
    bases at every 16-byte phase, 17 / 32 / 33 / 151 bases, second M-segments (the fast kernel's global X list) and
    clips on both ends.  The default context takes the window on the fast kernel; the forced one on the general kernel with
    packed-u8 low-BQ counters (copies = 1, fewer than 896 candidates) or one u32 per position (copies = 4)."""
    opt = CallableOptions(min_base_quality=min_bq)
    reads = H.quality_window(copies)
    assert (reads.n <= H.PACKED_LQ_READS) == (copies == 1)
    gw = run_three(contexts(opt), ("chrQ", 0, 3 * H.WREAL, H.reference(3 * H.WREAL, 3), reads), opt)
    assert gw == 0


def test_quality_bytes_in_a_deep_window(contexts):
    """More than 65535 short reads in one window: k_pileup_classify_deep, with BQ_HI."""
    opt = CallableOptions(max_depth=100_000, min_base_quality=129)
    reads = H.deep_quality_window()
    gw = run_three(contexts(opt), ("chrD", 0, 3 * H.WREAL, H.reference(3 * H.WREAL, 4), reads), opt)
    assert gw >= 1


# ------------------------------------------------------------------------------------------------ 3. threshold tables
def _staircase_case(contexts, fraction, opt, **kw):
    reads = H.staircase(fraction, **kw)
    length = H.staircase_len(fraction)
    gw = run_three(contexts(opt), ("chrS", 0, length, H.reference(length, 2), reads), opt)
    return gw, sum(1 for w in {s[3] for s in H.staircase_steps(fraction)}
                   if max(s[1] for s in H.staircase_steps(fraction) if s[3] == w) >= H.STAIR_SPLIT)


@pytest.mark.parametrize("fraction", H.FRACTIONS)
def test_low_mapq_thresholds_at_every_depth(contexts, fraction):
    """raw depths 1..300 with the low-MAPQ count at the threshold and one below it: the fast kernel's byte table (raw <= 254),
    the general kernel's shared-memory table (raw < 128) and the global table (128 and up) each decide some of them."""
    opt = CallableOptions(max_low_mapq_fraction=fraction)
    gw, deep_windows = _staircase_case(contexts, fraction, opt)
    assert deep_windows >= 1 and gw == deep_windows


@pytest.mark.parametrize("max_low_mapq", [0, 254, 255])
def test_low_mapq_thresholds_with_extreme_max_low_mapq(contexts, max_low_mapq):
    opt = CallableOptions(max_low_mapq=max_low_mapq, max_low_mapq_fraction=0.2)
    gw, deep_windows = _staircase_case(contexts, 0.2, opt, max_low_mapq=max_low_mapq, high_mapq=min(max_low_mapq + 1, 255))
    assert gw == deep_windows


def test_low_mapq_thresholds_with_min_mapping_quality_255(contexts):
    opt = CallableOptions(min_mapping_quality=255, max_low_mapq_fraction=1 / 3)
    gw, deep_windows = _staircase_case(contexts, 1 / 3, opt, high_mapq=255)
    assert gw == deep_windows


@pytest.mark.parametrize("min_depth,max_depth,min_dflm", [
    (0, 0, 0), (1, 1, 1), (U32_MAX, U32_MAX, U32_MAX), (0, U32_MAX, 1), (U32_MAX, 1, 0), (1, U32_MAX, U32_MAX), (2, 0, U32_MAX)])
def test_depth_options_at_their_u32_extremes(contexts, min_depth, max_depth, min_dflm):
    opt = CallableOptions(min_depth=min_depth, max_depth=max_depth, min_depth_for_low_mapq=min_dflm, max_low_mapq_fraction=0.1)
    gw, deep_windows = _staircase_case(contexts, 0.1, opt)
    assert gw == (0 if max_depth == 1 else deep_windows)      # max_depth 1 admits one read per start: no deep pile left


# ------------------------------------------------------------------------------------------------ 4. bail reasons
def _bail_case(contexts, reads, seed):
    return run_three(contexts(), ("chrB", 0, H.BAIL_LEN, H.reference(H.BAIL_LEN, seed), reads), CallableOptions())


@pytest.mark.parametrize("n_x", [H.F_XCAP, H.F_XCAP + 1])
def test_second_m_segments_at_the_cap(contexts, n_x):
    assert _bail_case(contexts, H.x_segment_window(n_x), 5) == (0 if n_x <= H.F_XCAP else 1)


@pytest.mark.parametrize("n_ops", [H.F_MAXOPS, H.F_MAXOPS + 1])
def test_cigar_ops_at_the_walk_limit(contexts, n_ops):
    assert _bail_case(contexts, H.ops_window(n_ops), 6) == (0 if n_ops <= H.F_MAXOPS else 1)


@pytest.mark.parametrize("n_cand", [H.N_CAND_FAST, H.N_CAND_FAST + 1])
def test_candidates_at_the_limit(contexts, n_cand):
    assert _bail_case(contexts, H.candidate_window(n_cand), 7) == (0 if n_cand <= H.N_CAND_FAST else 1)


@pytest.mark.parametrize("extra", [0, 1])
def test_cigar_density_at_the_rule(contexts, extra):
    assert _bail_case(contexts, H.density_window(extra), 8) == extra


@pytest.mark.parametrize("total", H.STAGE_TOTALS)
@pytest.mark.parametrize("phase", H.STAGE_PHASES)
def test_staged_quality_bytes_at_the_stage_size(contexts, total, phase):
    """k_window_ranges checks the staged bytes of every sub-batch with the same formula the fast kernel uses, so the fast
    kernel's own check never fails; what the limit decides is whether some sub-batch size of at least 4 reads fits.  Here
    the four long reads stage phase + total bytes, rounded up to 16: fast iff that is at most 4880."""
    fits = phase + total <= H.F_WSTAGE
    assert _bail_case(contexts, H.stage_window(total, phase), 9) == (0 if fits else 1)


def test_mixed_read_lengths_size_the_sub_batches(contexts):
    """Reads of 36..400 bases: the uniform-length shortcut of k_window_ranges does not apply and the shrink loop sizes
    the sub-batches.  Every window stays on the fast kernel."""
    length = 4 * H.WREAL
    gw = run_three(contexts(), ("chrL", 0, length, H.reference(length, 10), H.mixed_lengths()), CallableOptions())
    assert gw == 0


# ------------------------------------------------------------------------------------------------ 5. seams
@pytest.mark.parametrize("feature", H.SEAM_FEATURES)
def test_seams_between_fast_and_general_windows(contexts, feature):
    """Windows 2, 3 and 5 hold a 300-read pile: the kernels run fast, fast, general, general, fast, general, fast, fast,
    so the contig has every seam kind.  `feature` puts a REF_N run, a coverage gap or a depth / MAPQ step across,
    at the end of or at the start of every seam (or nothing: runs that continue through it)."""
    ref, reads = H.seam_contig(feature)
    gw = run_three(contexts(), ("chrZ", 0, H.SEAM_LEN, ref, reads), CallableOptions())
    assert gw == len(H.SEAM_PILES)


@pytest.mark.parametrize("feature", ["continue", "n_ends", "gap_starts", "depth_step"])
def test_region_shards_starting_at_seams(contexts, feature):
    """Region shards whose first window (always general) starts at a seam of the whole contig: fast -> general,
    general -> fast and fast -> general again.  Each shard matches the oracle per base, and the shards stitch to the whole."""
    opt = CallableOptions()
    ref, reads = H.seam_contig(feature)
    length = H.SEAM_LEN
    oc = run_oracle([("chrZ", 0, length, ref, reads)], opt, debug=True).contigs[0]
    adm = _admitted(reads, opt)
    span = adm.max_ref_span()
    end = adm.end()
    cuts = [0, 2 * H.WREAL, 4 * H.WREAL, 5 * H.WREAL, length]
    for ci, ctx in enumerate(contexts(opt)):
        parts = []
        for a, b in zip(cuts[:-1], cuts[1:]):
            sel = adm.select((adm.pos < b) & (end > a - 1))                  # the base left of the shard too
            ctx.begin_contig(0, "chrZ", length, ref, length, region=(a, b), max_ref_span=span)
            ctx.push_reads(sel)
            res = ctx.finish_contig()
            parts.append(res)
            raw, qc, low, st = ctx.debug_per_base(b - a)
            _same(f"raw [{a},{b})", raw, oc.raw[a:b]); _same(f"qc [{a},{b})", qc, oc.qc[a:b])
            _same(f"low [{a},{b})", low, oc.low[a:b]); _same(f"state [{a},{b})", st, oc.state[a:b])
            assert res.state_counts.tolist() == np.bincount(oc.state[a:b], minlength=6).tolist()
            assert res.n_covered_bases == int(np.count_nonzero(oc.raw[a:b]))
            assert res.summed_coverage == int(oc.raw[a:b].sum()) and res.quality_bases == int(oc.qc[a:b].sum())
            n_w = -(-(b - a) // H.WREAL)
            if ci == 0:
                plans = H.plan_windows(sel, length, region=(a, b), max_span=span)
                assert (plans[0].reason == "shard-first") == (a != 0) and res.general_windows == H.general_count(plans)
            else:
                assert res.general_windows == n_w
        iv = stitch_intervals([p.intervals for p in parts])
        want = states_to_intervals(oc.state)
        for f in ("start", "end", "state"):
            _same(f"stitched {f}", iv[f], want[f])
        for k in ("summed_baseq", "summed_mapq"):
            assert sum(getattr(p, k) for p in parts) == getattr(oc, k), k


# ------------------------------------------------------------------------------------------------ 6. synthetic contigs
@pytest.mark.parametrize("rl,depth", H.SYNTH_CASES)
def test_synthetic_contigs_of_other_read_lengths_and_depths(contexts, rl, depth):
    """Read lengths 36..250 at ordinary depths, and 150-base reads piled to 230x / 300x near the 254-read limit."""
    i = H.SYNTH_CASES.index((rl, depth))
    c = synth.synth_short("chr7", H.SYNTH_LEN, seed=900 + i, depth=depth, read_len=rl)
    gw = run_three(contexts(), (c.name, 0, c.length, c.ref, c.reads), CallableOptions())
    n_w = -(-c.length // H.WREAL)
    if depth >= 200:
        assert gw >= n_w - 2
    elif rl == 36:
        assert gw >= 1                     # windows with more than 96 second M-segments
    else:
        assert gw == 0


# ------------------------------------------------------------------------------------------------ refused batches
def _refuse(ctx, length, kind):
    """Push a batch that only the device can refuse (k_validate_batch) for a contig of `length` bases."""
    n = 64
    pos = np.linspace(5, max(length - 60, 6), n).astype(np.int32)
    coff = np.arange(n + 1, dtype=np.uint32)
    if kind == "unsorted":
        pos[n // 2], pos[n // 2 + 1] = pos[n // 2 + 1], pos[n // 2]
    else:
        coff[n // 2], coff[n // 2 + 1] = coff[n // 2 + 1], coff[n // 2]      # ends right, middle not monotone
    flag = np.zeros(n, np.uint16); mapq = np.full(n, 60, np.uint8); cig = np.full(n, (50 << 4), np.uint32)
    qoff = np.arange(n + 1, dtype=np.uint64) * 50; qual = np.full(n * 50, 30, np.uint8)
    keep = (pos, flag, mapq, coff, cig, qoff, qual)
    p = lambda a: a.ctypes.data
    ctx.begin_contig(0, "bad", length, b"A" * length, length, max_ref_span=50)
    ctx.push_raw(n, n, n * 50, *(p(a) for a in keep))
    with pytest.raises(ClbError):
        ctx.finish_contig()
    del keep


@pytest.mark.parametrize("forced", [False, True])
def test_refused_batches_leave_the_context_usable(forced):
    """A batch refused on the device leaves win_tab unwritten; the kernels after the pileup must not walk whatever an
    earlier contig (or no contig) left there.  Refused on a fresh context, right after a larger contig and right after a
    smaller one; each time the next good contig matches the oracle."""
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
        small = ("chrP", 0, H.DEPTH_LEN, H.reference(H.DEPTH_LEN, 1), H.depth_pile(254, 300))
        ref, reads = H.seam_contig("continue")
        large = ("chrZ", 0, H.SEAM_LEN, ref, reads)

        def good(contig):
            _check_context(ctx, contig, opt, run_oracle([contig], opt, debug=True).contigs[0])

        _refuse(ctx, 3 * H.WREAL, "unsorted")                      # fresh context: win_tab never written
        good(small)
        good(large)
        _refuse(ctx, H.WREAL - 7, "offsets")                       # after a larger contig
        good(small)
        _refuse(ctx, 6 * H.WREAL + 5, "unsorted")                  # after a smaller one: windows past its end
        good(large)
    finally:
        ctx.close()
