"""CPU checks of the hand-over inputs (tests/handover_inputs.py): the generators put every case on the side of its limit
that the GPU tests (tests/test_kernel_handover.py) expect, judged by the oracle's per-base counts and by the host model
of the window routing."""
import numpy as np
import pytest

from decodingustools_b200.options import CallableOptions
from oracle import oracle
from tests import handover_inputs as H
from tests.helpers import run_oracle


def _per_base(length, ref, reads, opt=None):
    return run_oracle([("c", 0, length, ref, reads)], opt or CallableOptions(), debug=True).contigs[0]


def _plans(reads, length, opt=None, **kw):
    opt = opt or CallableOptions()
    keep = oracle.admit(reads, opt.pileup_max_depth)
    assert keep.all(), "the generators' reads are all admitted"
    return H.plan_windows(reads, length, min_mapq=opt.min_mapping_quality, **kw)


@pytest.mark.parametrize("n_pile,n_before", [(254, 300), (254, 254), (255, 254), (255, 300)])
def test_depth_piles_are_exact_and_the_sample_missing_one_avoids_every_sample(n_pile, n_before):
    reads = H.depth_pile(n_pile, n_before)
    oc = _per_base(H.DEPTH_LEN, H.reference(H.DEPTH_LEN, 1), reads)
    assert int(oc.raw.max()) == n_pile and int(np.count_nonzero(oc.raw == n_pile)) == H.PILE_SPAN
    assert int(np.sort(oc.raw)[-H.PILE_SPAN - 1]) <= H.PILE_SPAN          # everywhere else: at most 50 reads
    span = reads.max_ref_span()
    assert span == H.PILE_SPAN
    r_lo = H.window_r_lo(reads.pos, 1, 0, span)
    r_hi = int(np.searchsorted(reads.pos, 2 * H.WREAL - 1 + H.WN - 1))
    a = H.pile_index(n_before)
    assert reads.pos[a] == reads.pos[a + n_pile - 1] and reads.pos[a - 1] < reads.pos[a]
    sampled = set(H.sample_indices(r_lo, r_hi))
    w1 = _plans(reads, H.DEPTH_LEN)[1]
    if n_pile == 254:
        assert not w1.read_deep and w1.path == "fast"
    elif n_before % 254:
        assert a + 254 not in sampled and not w1.sampled_deep               # no sample r_lo + 254 k lands on the pile's 255th read
        assert w1.read_deep and w1.reason == "read depth proof"
    else:
        assert a + 254 in sampled and w1.reason == "sampled depth proof"


@pytest.mark.parametrize("copies", [1, 4])
def test_quality_window_shapes_phases_and_layouts(copies):
    reads = H.quality_window(copies)
    plans = _plans(reads, 3 * H.WREAL)
    assert [p.path for p in plans] == ["fast", "fast", "fast"]
    assert (plans[1].n_cand <= H.PACKED_LQ_READS) == (copies == 1)
    assert 0 < plans[1].x_segments <= H.F_XCAP
    # every quality value of a segment base; every segment length 1..16 at every 16-byte phase of its first quality
    seen_q, seen_shape = set(), set()
    for i in range(reads.n):
        ops = reads.cigar[reads.cigar_off[i]:reads.cigar_off[i + 1]]
        q0, qp = int(reads.qual_off[i]), 0
        for v in ops:
            op, ln = int(v) & 15, int(v) >> 4
            if op == 0:
                seen_q.update(reads.qual[q0 + qp:q0 + qp + ln].tolist())
                seen_shape.add((ln, (q0 + qp) % 16))
            if op in (0, 1, 4):
                qp += ln
    assert seen_q == set(range(256))
    assert all((ln, a) in seen_shape for ln in range(1, 17) for a in range(16))
    assert all((ln, a) in seen_shape for ln in (17, 32, 33, 151) for a in (0, 1, 8, 15))


def test_deep_quality_window_goes_to_the_deep_kernel():
    reads = H.deep_quality_window()
    opt = CallableOptions(max_depth=100_000)
    plans = _plans(reads, 3 * H.WREAL, opt)
    assert plans[1].n_cand > H.DEEP_CAND and plans[1].path == "deep"


@pytest.mark.parametrize("fraction", H.FRACTIONS)
def test_staircase_has_the_intended_raw_and_low_at_every_position(fraction):
    reads = H.staircase(fraction)
    steps = H.staircase_steps(fraction)
    length = H.staircase_len(fraction)
    oc = _per_base(length, H.reference(length, 2), reads)
    want_raw = np.zeros(length, np.uint32); want_low = np.zeros(length, np.uint32)
    for p, raw, low, _ in steps:
        want_raw[p] = raw; want_low[p] = low
    assert np.array_equal(oc.raw, want_raw) and np.array_equal(oc.low, want_low)
    # each step sits at the threshold or just below it; the raw runs cross every table seam
    for p, raw, low, _ in steps:
        t = H.first_low(raw, fraction)
        assert low in (t - 1, t) or low == raw
    raws = {s[1] for s in steps}
    assert {1, H.NFIRST - 1, H.NFIRST, 254, 255, 256, 300} <= raws
    # windows of depths <= 254 are fast, the ones from 255 on general
    deepest = {}
    for p, raw, low, w in steps:
        deepest[w] = max(deepest.get(w, 0), raw)
    plans = _plans(reads, length)
    assert [p.path for p in plans] == ["fast" if deepest.get(p.w, 0) < H.STAIR_SPLIT else "general" for p in plans]
    assert {"fast", "general"} <= {p.path for p in plans}


@pytest.mark.parametrize("n_x", [H.F_XCAP, H.F_XCAP + 1])
def test_x_segment_counts_sit_on_both_sides_of_the_cap(n_x):
    w1 = _plans(H.x_segment_window(n_x), H.BAIL_LEN)[1]
    assert w1.x_segments == n_x and w1.max_ops == 3 and not w1.read_deep
    assert w1.path == ("fast" if n_x <= H.F_XCAP else "general")


@pytest.mark.parametrize("n_ops", [H.F_MAXOPS, H.F_MAXOPS + 1])
def test_op_counts_sit_on_both_sides_of_the_walk_limit(n_ops):
    w1 = _plans(H.ops_window(n_ops), H.BAIL_LEN)[1]
    assert w1.max_ops == n_ops and w1.n_ops <= 8 * w1.n_cand + 64 and w1.x_segments == (1 if n_ops <= H.F_MAXOPS else 0)
    assert w1.reason == (None if n_ops <= H.F_MAXOPS else "ops")


@pytest.mark.parametrize("n_cand", [H.N_CAND_FAST, H.N_CAND_FAST + 1])
def test_candidate_counts_sit_on_both_sides_of_the_limit(n_cand):
    w1 = _plans(H.candidate_window(n_cand), H.BAIL_LEN)[1]
    assert w1.n_cand == n_cand
    assert w1.reason == (None if n_cand <= H.N_CAND_FAST else "candidates")


@pytest.mark.parametrize("extra", [0, 1])
def test_cigar_density_sits_on_both_sides_of_the_rule(extra):
    w1 = _plans(H.density_window(extra), H.BAIL_LEN)[1]
    assert w1.n_cand == 16 and w1.n_ops == 8 * 16 + 64 + extra and w1.max_ops <= H.F_MAXOPS and w1.x_segments == 16
    assert w1.reason == (None if extra == 0 else "cigar density")


@pytest.mark.parametrize("total", H.STAGE_TOTALS)
@pytest.mark.parametrize("phase", H.STAGE_PHASES)
def test_stage_bytes_sit_on_the_intended_side(total, phase):
    reads = H.stage_window(total, phase)
    w1 = _plans(reads, H.BAIL_LEN)[1]
    assert int(reads.qual_off[w1.r_lo]) % 16 == phase and int(reads.qual_off[w1.r_lo + 4] - reads.qual_off[w1.r_lo]) == total
    assert w1.shrunk
    if phase + total <= H.F_WSTAGE:
        assert w1.path == "fast" and w1.G in (4, 5)
    else:
        assert w1.reason == "stage"


def test_mixed_lengths_need_the_shrink_loop():
    plans = _plans(H.mixed_lengths(), 4 * H.WREAL)
    assert any(p.shrunk for p in plans) and all(p.path == "fast" for p in plans)


@pytest.mark.parametrize("feature", H.SEAM_FEATURES)
def test_seam_contig_kernel_sequence_and_seam_states(feature):
    ref, reads = H.seam_contig(feature)
    plans = _plans(reads, H.SEAM_LEN)
    assert "".join("G" if p.reason else "F" for p in plans) == "FFGGFGFF"
    oc = _per_base(H.SEAM_LEN, ref, reads)
    seams = [w * H.WREAL for w in range(1, H.SEAM_WINDOWS)]
    st = oc.state
    if feature == "continue":
        assert sum(st[s - 1] == st[s] for s in seams) >= 5
    elif feature in ("n_through", "n_ends", "n_starts", "gap_ends", "gap_starts", "depth_step"):
        for s in seams:
            changes = {"n_through": False, "n_ends": True, "n_starts": True, "gap_ends": True, "gap_starts": True, "depth_step": True}[feature]
            assert (st[s - 1] != st[s]) == changes, (feature, s, st[s - 1], st[s])
    elif feature == "gap_through":
        assert all(st[s - 1] == st[s] == 2 for s in seams)                   # NO_COVERAGE through the seam


@pytest.mark.parametrize("rl,depth", H.SYNTH_CASES)
def test_synthetic_contigs_route_as_expected(rl, depth):
    from decodingustools_b200 import synth
    i = H.SYNTH_CASES.index((rl, depth))
    c = synth.synth_short("chr7", H.SYNTH_LEN, seed=900 + i, depth=depth, read_len=rl)
    reads = c.reads.select(oracle.admit(c.reads, 500))
    plans = H.plan_windows(reads, c.length)
    reasons = {p.reason for p in plans}
    if depth >= 200:                               # piles past 254 reads: almost every window fails the sampled depth proof
        assert H.general_count(plans) >= len(plans) - 2 and "sampled depth proof" in reasons
    elif rl == 36:                                 # many short indel reads: windows with more than 96 second M-segments
        assert reasons == {None, "x segments"}
    else:
        assert reasons == {None}
