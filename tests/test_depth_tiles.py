"""Depth tiles (clb_set_depth_tiles / CallableLociContext.set_depth_tiles): per fixed-size tile of a contig, the positions
that are not REF_N (territory), the CALLABLE ones and the raw / QC depth sums over the territory, counted in phase C of all
three pileup kernels, against the oracle's per-base dump summed over each tile.

Every kernel case runs in a default context (fast kernel for ordinary windows) and in a CLB_FORCE_GENERAL=1 context (every
window through the general kernel), at tile lengths on both sides of a warp (256 entries) and of a window (2047
positions), longer than the contig, and the largest one allowed."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from decodingustools_b200 import synth
from decodingustools_b200._lib import ClbError
from decodingustools_b200.callable_loci import CallableLociContext, admit_reads, compact_reads, depth_tile_ranges
from decodingustools_b200.options import CallableOptions
from decodingustools_b200.sharding import pack_counters, unpack_counters
from tests import bamio
from tests import handover_inputs as H
from tests.helpers import assert_parity, run_oracle

pytestmark = pytest.mark.gpu

LS = (256, 257, 1000, 2047, 2048, 4094, 10007, 1_000_000, 2**31)
REF_N, CALLABLE = 0, 1
FIELDS = ("tile_territory", "tile_callable", "tile_raw_sum", "tile_qc_sum")
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


def expected(oc, length, tile_len, lo=0, hi=None):
    """Oracle tiles (territory, callable, raw_sum, qc_sum) of positions [lo, hi) from its per-base dump."""
    hi = length if hi is None else hi
    n = len(depth_tile_ranges(length, tile_len)[0])
    t = np.arange(lo, hi, dtype=np.int64) // tile_len
    state = np.asarray(oc.state[lo:hi])
    own = state != REF_N
    out = [np.bincount(t[own], minlength=n).astype(np.uint64), np.bincount(t[state == CALLABLE], minlength=n).astype(np.uint64)]
    for depth in (oc.raw, oc.qc):
        s = np.zeros(n, np.uint64)
        np.add.at(s, t[own], np.asarray(depth[lo:hi])[own].astype(np.uint64))
        out.append(s)
    return out


def _same(what, got, want):
    assert got is not None, what
    got, want = np.asarray(got, np.uint64), np.asarray(want).astype(np.uint64)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    bad = np.flatnonzero(got != want)
    assert bad.size == 0, f"{what}: {bad.size} tiles differ, first {bad[0]}: got {got[bad[0]]}, want {want[bad[0]]}"


def check_tiles(what, res, want):
    for f, w in zip(FIELDS, want):
        _same(f"{what} {f}", getattr(res, f), w)


def check_invariants(res, region_len):
    assert int(res.tile_territory.sum()) == region_len - int(res.state_counts[REF_N])
    assert int(res.tile_callable.sum()) == int(res.state_counts[CALLABLE])
    if res.depth_hist_raw is not None:
        n = len(res.depth_hist_raw)
        d = np.arange(n, dtype=np.uint64)
        if res.depth_hist_raw[n - 1] == 0:                                 # no clamped depth: the histogram sums follow
            assert int(res.tile_raw_sum.sum()) == int((d * res.depth_hist_raw).sum())
        if res.depth_hist_qc[n - 1] == 0:
            assert int(res.tile_qc_sum.sum()) == int((d * res.depth_hist_qc).sum())


def run_case(pair, contig, opt, ls=LS, hist=0):
    """Both contexts, every tile length: assert_parity with the tiles on (BED, counts, sums, bins, export), tiles equal to
    the oracle's, the invariants, and the counter buffer's length."""
    name, tid, length, ref, reads = contig
    oc = run_oracle([contig], opt, debug=True).contigs[0]
    for ctx in pair:
        ctx.set_depth_histogram(hist)
        for L in ls:
            ctx.set_depth_tiles(L)
            _, results = assert_parity([contig], opt, ctx)
            res = results[0]
            n = len(depth_tile_ranges(length, L)[0])
            assert res.tile_len == L and len(res.tile_territory) == n
            check_tiles(f"L={L}", res, expected(oc, length, L))
            check_invariants(res, length)
            assert ctx.counters_device()[1] == 12 + 3 * res.bins.shape[1] + 2 * hist + 4 * n
        ctx.set_depth_tiles(0)
        ctx.set_depth_histogram(0)
    return oc


def tile_edge_contig(tile_len, seed=43):
    """The 8-window hand-over contig (300-read piles in windows 2, 3 and 5: fast, fast, general, general, fast, general,
    fast, fast) with REF_N runs that end and start on tile boundaries and depth steps on them: 80 reads end and 40 MAPQ-0
    reads start at every boundary."""
    rng = np.random.default_rng(seed)
    edges = list(range(tile_len, H.SEAM_LEN, tile_len))
    n_runs = [(e - 9, e) for e in edges[0::3]] + [(e, e + 9) for e in edges[1::3]]
    ref = H.reference(H.SEAM_LEN, seed, n_runs)
    starts = list(np.sort(rng.integers(0, H.SEAM_LEN - 100, int(12 * H.SEAM_LEN / 100))))
    mapq = list(rng.choice([60, 60, 60, 30, 0], size=len(starts)))
    for e in edges:
        starts += [e - 100] * 80; mapq += [60] * 80
        if e + 100 <= H.SEAM_LEN:
            starts += [e] * 40; mapq += [0] * 40
    for w in H.SEAM_PILES:
        starts += [w * H.WREAL + 1000] * 300; mapq += [60] * 300
    order = np.argsort(np.array(starts), kind="stable")
    pos = [int(starts[i]) for i in order]
    mq = np.array([mapq[i] for i in order], np.uint8)
    return ref, H.columns(pos, ["100M"] * len(pos), mq, H.rotating_quals([100] * len(pos), step=19))


# ------------------------------------------------------------------------------------------------ kernel coverage
def test_synthetic_30x_contig(contexts):
    c = synth.synth_short("chr9", 300_000, seed=77)
    run_case(contexts(CallableOptions()), (c.name, 0, c.length, c.ref, c.reads), CallableOptions())


@pytest.mark.parametrize("tile_len", [256, 1000, 2047])
def test_hand_over_contig_with_ref_n_and_depth_steps_on_tile_boundaries(contexts, tile_len):
    ref, reads = tile_edge_contig(tile_len)
    oc = run_case(contexts(CallableOptions()), ("chrZ", 0, H.SEAM_LEN, ref, reads), CallableOptions(), ls=(tile_len,))
    assert int(oc.counts[REF_N]) > 0


@pytest.mark.parametrize("feature", ["n_through", "n_ends", "n_starts", "depth_step"])
def test_hand_over_contig_with_features_at_window_seams(contexts, feature):
    """L = 2047: every tile boundary is a window seam."""
    ref, reads = H.seam_contig(feature)
    run_case(contexts(CallableOptions()), ("chrZ", 0, H.SEAM_LEN, ref, reads), CallableOptions(), ls=(256, 2047, 4094))


def test_deep_window(contexts):
    """More than 65535 candidates in one window: k_pileup_classify_deep (64-bit depth sums)."""
    opt = CallableOptions(max_depth=100_000, min_base_quality=129)
    run_case(contexts(opt), ("chrD", 0, 3 * H.WREAL, H.reference(3 * H.WREAL, 4), H.deep_quality_window()), opt,
             ls=(256, 1000, 2047, 2**31))


def test_long_read_contig(contexts):
    c = synth.synth_long("chr2", 120_000, seed=78, depth=20.0)
    run_case(contexts(CallableOptions()), (c.name, 0, c.length, c.ref, c.reads), CallableOptions(), ls=(256, 1000, 10007))


def test_2000x_pile(contexts):
    """Depths well past the fast kernel's 254 and the general kernel's 16-bit packing of a warp's 256 entries."""
    opt = CallableOptions(max_depth=4000)
    c = synth.synth_short("chrY", 12_000, seed=4, depth=2000.0)
    oc = run_case(contexts(opt), (c.name, 0, c.length, c.ref, c.reads), opt, ls=(256, 1000, 2047))
    assert int(oc.raw.max()) > 1000


def test_tiles_and_histograms_together(contexts):
    c = synth.synth_short("chr3", 200_000, seed=83)
    run_case(contexts(CallableOptions()), (c.name, 0, c.length, c.ref, c.reads), CallableOptions(), ls=(256, 1000, 2047), hist=1001)


# ------------------------------------------------------------------------------------------------ region shards
def test_region_shards_sum_to_the_whole_contig(contexts):
    """Shards cut at window multiples (their first windows are general, with the halo entry) add into the same
    whole-contig tiles, and pack_counters / unpack_counters carry them."""
    opt = CallableOptions()
    ref, reads = H.seam_contig("depth_step")                           # the halo positions carry depth
    length = H.SEAM_LEN
    oc = run_oracle([("chrZ", 0, length, ref, reads)], opt, debug=True).contigs[0]
    adm = compact_reads(reads, admit_reads(reads, opt.pileup_max_depth, 0))
    span, end = adm.max_ref_span(), adm.end()
    cuts = [0, 2 * H.WREAL, 4 * H.WREAL, 5 * H.WREAL, length]
    for ctx in contexts(opt):
        for L in (256, 1000, 3000):
            ctx.set_depth_tiles(L)
            parts = []
            for a, b in zip(cuts[:-1], cuts[1:]):
                ctx.begin_contig(0, "chrZ", length, ref, length, region=(a, b), max_ref_span=span)
                ctx.push_reads(adm.select((adm.pos < b) & (end > a - 1)))
                res = ctx.finish_contig()
                check_tiles(f"L={L} shard [{a},{b})", res, expected(oc, length, L, a, b))
                check_invariants(res, b - a)
                parts.append(res)
            vec = sum(pack_counters(p).view(np.uint64) for p in parts)
            whole = unpack_counters(vec.view(np.int64), parts[0])
            check_tiles(f"L={L} summed", whole, expected(oc, length, L))
            assert whole.state_counts.tolist() == oc.counts and whole.summed_coverage == oc.summed_coverage
        ctx.set_depth_tiles(0)


# ------------------------------------------------------------------------------------------------ repeated and re-run work
def test_reruns_debug_runs_and_refresh_return_the_same_tiles(contexts):
    opt = CallableOptions()
    c = synth.synth_short("chr4", 100_000, seed=79)
    contig = (c.name, 0, c.length, c.ref, c.reads)
    oc = run_oracle([contig], opt, debug=True).contigs[0]
    want = expected(oc, c.length, 1000)
    for ctx in contexts(opt):
        ctx.set_depth_tiles(1000)
        _, results = assert_parity([contig], opt, ctx)
        first = results[0]
        _, r1 = ctx.rerun_resident(fetch=True)
        _, r2 = ctx.rerun_resident(fetch=True)
        ctx.debug_per_base(c.length)
        r3 = ctx.refresh_counters()
        for what, r in (("finish", first), ("rerun 1", r1), ("rerun 2", r2), ("refresh after debug", r3)):
            check_tiles(what, r, want)
        ctx.set_depth_tiles(0)


def test_record_capacity_rerun_keeps_the_tiles(contexts):
    """REF_N at every other position: more run starts than the first record buffer holds, so clb_finish_contig grows it and
    re-runs the contig from reset accumulators."""
    opt = CallableOptions()
    length = 120_000
    ref = bytearray(H.reference(length, 12))
    ref[1:100_000:2] = b"N" * len(range(1, 100_000, 2))
    c = synth.synth_short("chrR", length, seed=80, depth=12.0)
    run_case(contexts(opt), ("chrR", 0, length, bytes(ref), c.reads), opt, ls=(256, 1000))


# ------------------------------------------------------------------------------------------------ switching and errors
def test_switching_the_tile_length_and_turning_tiles_off_between_contigs(contexts):
    opt = CallableOptions()
    c = synth.synth_short("chr5", 60_000, seed=81)
    contig = (c.name, 0, c.length, c.ref, c.reads)
    oc = run_oracle([contig], opt, debug=True).contigs[0]
    for ctx in contexts(opt):
        ctx.set_depth_tiles(0)
        _, off = assert_parity([contig], opt, ctx)
        for L in (5000, 256, 70_000):
            ctx.set_depth_tiles(L)
            _, on = assert_parity([contig], opt, ctx)
            check_tiles(f"L={L}", on[0], expected(oc, c.length, L))
            assert np.array_equal(on[0].intervals, off[0].intervals) and np.array_equal(on[0].bins, off[0].bins)
            assert on[0].state_counts.tolist() == off[0].state_counts.tolist()
        ctx.set_depth_tiles(0)
        _, off2 = assert_parity([contig], opt, ctx)
        assert all(getattr(off2[0], f) is None for f in FIELDS) and off2[0].tile_len == 0
        assert ctx.counters_device()[1] == 12 + 3 * off2[0].bins.shape[1]
        _, rr = ctx.rerun_resident(fetch=True)
        assert rr.tile_territory is None


def test_invalid_settings_are_refused(contexts):
    opt = CallableOptions()
    ctx = contexts(opt)[0]
    for L in (1, 255, 2**31 + 1):
        with pytest.raises(ClbError) as e:
            ctx.set_depth_tiles(L)
        assert e.value.code == -1
    c = synth.synth_short("chr6", 20_000, seed=82)
    ctx.begin_contig(0, c.name, c.length, c.ref, c.length)
    with pytest.raises(ClbError) as e:
        ctx.set_depth_tiles(1000)
    assert e.value.code == -1
    ctx.push_reads(compact_reads(c.reads, admit_reads(c.reads, opt.pileup_max_depth, 0)))
    assert ctx.finish_contig().tile_territory is None
    ctx.set_depth_tiles(0)


# ------------------------------------------------------------------------------------------------ coverage command
def expected_tsv(ocs, tile_len):
    lines = ["#contig\tstart\tend\tterritory\tcallable\tmean_raw\tmean_qc"]
    for oc in ocs:
        length = oc.length
        ter, cal, raw, qc = expected(oc, length, tile_len)
        for t, (s, e) in enumerate(zip(*depth_tile_ranges(length, tile_len))):
            mr = int(raw[t]) / int(ter[t]) if ter[t] else 0.0
            mq = int(qc[t]) / int(ter[t]) if ter[t] else 0.0
            lines.append(f"{oc.name}\t{s}\t{e}\t{int(ter[t])}\t{int(cal[t])}\t{mr:.2f}\t{mq:.2f}")
    return "\n".join(lines) + "\n"


def _outputs(d):
    return {p: (d / p).read_bytes() for p in sorted(os.listdir(d)) if p.endswith((".bed", ".json", ".html", ".svg"))}


def _cli(cwd, args):
    return subprocess.run([CLI, "coverage", *args], cwd=cwd, capture_output=True, text=True, timeout=600)


@pytest.mark.parametrize("size", [None, 256, 50_000])
def test_cli_tiles_of_a_small_genome(tmp_path, size):
    cs = [synth.synth_short("chr1", 120_000, seed=41), synth.synth_short("chr2", 60_000, seed=42),
          synth.synth_short("chrM", 16_569, seed=43, depth=300.0)]
    contigs = [(c.name, tid, c.length, c.ref, c.reads) for tid, c in enumerate(cs)]
    (tmp_path / "off").mkdir(); (tmp_path / "on").mkdir()
    bam = str(tmp_path / "in.bam"); fa = str(tmp_path / "ref.fa")
    bamio.write_bam(bam, [(n, l, r) for n, _, l, _, r in contigs])
    bamio.write_fasta(fa, [(n, ref) for n, _, _, ref, _ in contigs])
    off = _cli(tmp_path / "off", [bam, "-r", fa, "-o", "out.bed"])
    extra = [] if size is None else ["--depth-tile-size", str(size)]
    on = _cli(tmp_path / "on", [bam, "-r", fa, "-o", "out.bed", "--depth-tiles", "tiles.tsv", *extra])
    assert off.returncode == 0 and on.returncode == 0, (off.stderr, on.stderr)
    assert _outputs(tmp_path / "on") == _outputs(tmp_path / "off") and len(_outputs(tmp_path / "off")) >= 5
    ocs = run_oracle(contigs, CallableOptions(), debug=True).contigs
    assert (tmp_path / "on" / "tiles.tsv").read_text() == expected_tsv(ocs, size or 1000)


def test_cli_tiles_of_the_deep_golden_case(tmp_path):
    """mini_config4_deep_cap500 with tiles and the depth histogram on: the golden outputs stay byte-identical."""
    from tests.golden_cases import cases
    name = "mini_config4_deep_cap500"
    for f in ("in.bam", "in.bam.bai", "ref.fa", "ref.fa.fai"):
        shutil.copy(os.path.join(GOLDEN, name, f), tmp_path / f)
    p = _cli(tmp_path, ["in.bam", "-r", "ref.fa", "-o", "callable_regions.bed", "--depth-tiles", "t.tsv", "--depth-tile-size", "300",
                        "--depth-histogram", "h.tsv"])
    assert p.returncode == 0, p.stderr
    assert (tmp_path / "callable_regions.bed").read_bytes() == open(os.path.join(GOLDEN, name, "expected.callable_regions.bed"), "rb").read()
    assert (tmp_path / "summary.json").read_text() == open(os.path.join(GOLDEN, name, "expected.summary.json")).read()
    _, contigs, opt = next(c for c in cases() if c[0] == name)
    ocs = run_oracle([(n, tid, l, ref, r) for tid, (n, l, ref, r) in enumerate(contigs)], opt, debug=True).contigs
    assert (tmp_path / "t.tsv").read_text() == expected_tsv(ocs, 300)


def test_cli_bad_tile_size_and_unwritable_tiles_path(tmp_path):
    c = synth.synth_short("chr1", 30_000, seed=44)
    bam = str(tmp_path / "in.bam"); fa = str(tmp_path / "ref.fa")
    bamio.write_bam(bam, [(c.name, c.length, c.reads)]); bamio.write_fasta(fa, [(c.name, c.ref)])
    for bad in ("255", str(2**31 + 1)):
        p = _cli(tmp_path, [bam, "-r", fa, "-o", "out.bed", "--depth-tiles", "t.tsv", "--depth-tile-size", bad])
        assert p.returncode == 2 and "--depth-tile-size" in p.stderr
    (tmp_path / "t.tsv").mkdir()
    p = _cli(tmp_path, [bam, "-r", fa, "-o", "out.bed", "--depth-tiles", str(tmp_path / "t.tsv")])
    assert p.returncode == 1, p.stderr[-2000:]
    assert p.stderr.splitlines()[-1] == f"Error: cannot write {tmp_path / 't.tsv'}", p.stderr[-2000:]
