"""Depth thresholds per tile (clb_set_depth_thresholds / CallableLociContext.set_depth_thresholds): per depth tile and
threshold T_j, the positions that are not REF_N with raw (QC) depth >= T_j, counted in phase C of all three pileup kernels,
against the oracle's per-base dump binned per tile.

Every kernel case runs in a default context (fast kernel for ordinary windows) and in a CLB_FORCE_GENERAL=1 context (every
window through the general kernel), with assert_parity, the tiles and the threshold invariants."""
import os
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
from tests.test_depth_runs import deep_pile
from tests.test_depth_tiles import check_tiles, expected as expected_tiles, expected_tsv, tile_edge_contig

pytestmark = pytest.mark.gpu

LS = (256, 257, 2047, 2048, 10007, 2**31)
K8 = (1, 4, 10, 20, 30, 40, 60, 100)                                  # 4: min_depth
REF_N = 0
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLI = os.path.join(ROOT, "decodingustools_b200", "decodingus-tools-b200")


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


def expected(oc, length, tile_len, thresholds, lo=0, hi=None):
    """Oracle (raw_ge, qc_ge), [K, n_tiles] each, of positions [lo, hi) from its per-base dump."""
    hi = length if hi is None else hi
    n = len(depth_tile_ranges(length, tile_len)[0])
    t = np.arange(lo, hi, dtype=np.int64) // tile_len
    own = np.asarray(oc.state[lo:hi]) != REF_N
    out = []
    for depth in (oc.raw, oc.qc):
        d = np.asarray(depth[lo:hi]).astype(np.int64)
        out.append(np.array([np.bincount(t[own & (d >= T)], minlength=n) for T in thresholds], np.uint64).reshape(len(thresholds), n))
    return out


def check_ge(what, res, thresholds, want):
    assert res.tile_thresholds is not None and res.tile_thresholds.tolist() == list(thresholds), what
    for name, got, w in (("raw_ge", res.tile_raw_ge, want[0]), ("qc_ge", res.tile_qc_ge, want[1])):
        assert got.shape == w.shape, (what, name, got.shape, w.shape)
        bad = np.argwhere(got != w)
        assert bad.size == 0, f"{what} {name}: {len(bad)} counts differ, first [j={bad[0][0]}, tile {bad[0][1]}]: got {got[tuple(bad[0])]}, want {w[tuple(bad[0])]}"


def check_invariants(res):
    raw, qc, ter = res.tile_raw_ge.astype(np.int64), res.tile_qc_ge.astype(np.int64), res.tile_territory.astype(np.int64)
    assert np.all(raw <= ter) and np.all(qc <= raw)
    assert np.all(np.diff(raw, axis=0) <= 0) and np.all(np.diff(qc, axis=0) <= 0)
    if res.depth_hist_raw is not None:
        n = len(res.depth_hist_raw)
        for j, T in enumerate(res.tile_thresholds.tolist()):
            if res.depth_hist_raw[n - 1] == 0:                             # no clamped depth: the histogram's tail follows
                assert int(raw[j].sum()) == int(res.depth_hist_raw[min(T, n):].sum())
            if res.depth_hist_qc[n - 1] == 0:
                assert int(qc[j].sum()) == int(res.depth_hist_qc[min(T, n):].sum())


def run_case(pair, contig, opt, thresholds_list=((10,), K8), ls=LS, hist=0, runs=False, oc=None):
    """Both contexts, every threshold list and tile length: assert_parity, tiles and threshold counts equal to the oracle's,
    the invariants, and the counter buffer's length."""
    name, tid, length, ref, reads = contig
    oc = oc or run_oracle([contig], opt, debug=True).contigs[0]
    for ctx in pair:
        ctx.set_depth_histogram(hist)
        ctx.set_depth_runs(runs)
        for thresholds in thresholds_list:
            ctx.set_depth_thresholds(thresholds)
            for L in ls:
                ctx.set_depth_tiles(L)
                _, results = assert_parity([contig], opt, ctx)
                res = results[0]
                n = len(depth_tile_ranges(length, L)[0])
                check_tiles(f"L={L}", res, expected_tiles(oc, length, L))
                check_ge(f"T={thresholds} L={L}", res, thresholds, expected(oc, length, L, thresholds))
                check_invariants(res)
                assert ctx.counters_device()[1] == 12 + 3 * res.bins.shape[1] + 2 * hist + (4 + 2 * len(thresholds)) * n
        ctx.set_depth_thresholds(())
        ctx.set_depth_tiles(0)
        ctx.set_depth_histogram(0)
        ctx.set_depth_runs(False)
    return oc


# ------------------------------------------------------------------------------------------------ kernel coverage
def test_synthetic_30x_contig(contexts):
    c = synth.synth_short("chr9", 300_000, seed=77)
    oc = run_case(contexts(CallableOptions()), (c.name, 0, c.length, c.ref, c.reads), CallableOptions())
    raw, qc = expected(oc, c.length, 1000, K8)
    assert not np.array_equal(raw, qc)                                  # raw and QC differ: a swap of the kinds shows


@pytest.mark.parametrize("tile_len", [256, 1000, 2047])
def test_hand_over_contig_with_ref_n_and_depth_steps_on_tile_boundaries_and_thresholds(contexts, tile_len):
    """Depth steps on every tile boundary (80 reads end, 40 MAPQ-0 reads start), REF_N runs under reads that end and start
    on boundaries, and thresholds equal to the depths on both sides of the boundaries."""
    ref, reads = tile_edge_contig(tile_len)
    contig = ("chrZ", 0, H.SEAM_LEN, ref, reads)
    opt = CallableOptions()
    oc = run_oracle([contig], opt, debug=True).contigs[0]
    edges = np.arange(tile_len, H.SEAM_LEN, tile_len)
    at = sorted({int(oc.raw[e]) for e in edges} | {int(oc.raw[e - 1]) for e in edges} | {int(oc.qc[e]) for e in edges})
    picks = tuple(at[:: max(1, len(at) // 8)][:8])
    assert int(oc.counts[REF_N]) > 0 and len(picks) >= 4
    run_case(contexts(opt), contig, opt, thresholds_list=(picks,), ls=(tile_len,), oc=oc)


@pytest.mark.parametrize("feature", ["n_through", "depth_step"])
def test_hand_over_contig_with_features_at_window_seams(contexts, feature):
    ref, reads = H.seam_contig(feature)
    run_case(contexts(CallableOptions()), ("chrZ", 0, H.SEAM_LEN, ref, reads), CallableOptions(), thresholds_list=(K8,),
             ls=(256, 2047))


def test_deep_window_at_and_above_its_max_depth(contexts):
    """More than 65535 candidates in one window: k_pileup_classify_deep compares full 32-bit depths."""
    opt = CallableOptions(max_depth=100_000, min_base_quality=129)
    contig = ("chrD", 0, 3 * H.WREAL, H.reference(3 * H.WREAL, 4), H.deep_quality_window())
    oc = run_oracle([contig], opt, debug=True).contigs[0]
    top, qtop = int(oc.raw.max()), int(oc.qc.max())
    ths = tuple(sorted({1, 255, 65536, qtop, top - 1, top, top + 1, 2**32 - 1}))
    run_case(contexts(opt), contig, opt, thresholds_list=(ths,), ls=(256, 2047, 2**31), oc=oc)


def test_deep_pile_past_16_bits(contexts):
    """Raw depths past 65535, which only the deep kernel's 32-bit depth arrays hold: thresholds on both sides of 2^16."""
    opt = CallableOptions(max_depth=100_000)
    contig = ("chrP", 0, 3 * H.WREAL, H.reference(3 * H.WREAL, 6), deep_pile())
    oc = run_oracle([contig], opt, debug=True).contigs[0]
    top = int(oc.raw.max())
    assert top > 65536
    run_case(contexts(opt), contig, opt, thresholds_list=((1, 255, 256, 65535, 65536, top, top + 1),), ls=(256, 2047), oc=oc)


def test_long_read_contig(contexts):
    c = synth.synth_long("chr2", 120_000, seed=78, depth=20.0)
    run_case(contexts(CallableOptions()), (c.name, 0, c.length, c.ref, c.reads), CallableOptions(), thresholds_list=(K8,),
             ls=(256, 10007))


def test_2000x_pile_around_the_fast_kernels_byte_ceiling(contexts):
    opt = CallableOptions(max_depth=4000)
    c = synth.synth_short("chrY", 12_000, seed=4, depth=2000.0)
    oc = run_case(contexts(opt), (c.name, 0, c.length, c.ref, c.reads), opt,
                  thresholds_list=((253, 254, 255, 256, 257, 1000, 1500, 2000), (254,), (255,)), ls=(256, 2047))
    assert int(oc.raw.max()) > 1000


def test_all_four_features_together_and_debug_equals_production(contexts):
    """Feature set 15 (histograms, tiles, runs, thresholds); the per-base debug run (DBG instantiations) refreshes the same
    counters as the production run."""
    opt = CallableOptions()
    c = synth.synth_short("chr3", 200_000, seed=83)
    contig = (c.name, 0, c.length, c.ref, c.reads)
    oc = run_case(contexts(opt), contig, opt, thresholds_list=(K8,), ls=(256, 1000), hist=1001, runs=True)
    for ctx in contexts(opt):
        ctx.set_depth_histogram(1001); ctx.set_depth_runs(True); ctx.set_depth_tiles(1000); ctx.set_depth_thresholds(K8)
        _, results = assert_parity([contig], opt, ctx)
        first = results[0]
        ctx.debug_per_base(c.length)
        again = ctx.refresh_counters()
        check_ge("debug run", again, K8, expected(oc, c.length, 1000, K8))
        assert np.array_equal(again.tile_raw_ge, first.tile_raw_ge) and np.array_equal(again.tile_qc_ge, first.tile_qc_ge)
        assert np.array_equal(again.depth_hist_raw, first.depth_hist_raw) and np.array_equal(again.depth_runs, first.depth_runs)
        ctx.set_depth_thresholds(()); ctx.set_depth_tiles(0); ctx.set_depth_runs(False); ctx.set_depth_histogram(0)


# ------------------------------------------------------------------------------------------------ region shards
def test_region_shards_with_the_halo_on_a_tile_boundary_sum_to_the_whole_contig(contexts):
    """Shards cut at window multiples (their first windows are general, with the halo entry, which carries depth); at
    L = 2047 every cut is also a tile boundary."""
    opt = CallableOptions()
    ref, reads = H.seam_contig("depth_step")
    length = H.SEAM_LEN
    oc = run_oracle([("chrZ", 0, length, ref, reads)], opt, debug=True).contigs[0]
    adm = compact_reads(reads, admit_reads(reads, opt.pileup_max_depth, 0))
    span, end = adm.max_ref_span(), adm.end()
    cuts = [0, 2 * H.WREAL, 4 * H.WREAL, 5 * H.WREAL, length]
    for ctx in contexts(opt):
        ctx.set_depth_thresholds(K8)
        for L in (2047, 256, 1000):
            ctx.set_depth_tiles(L)
            parts = []
            for a, b in zip(cuts[:-1], cuts[1:]):
                ctx.begin_contig(0, "chrZ", length, ref, length, region=(a, b), max_ref_span=span)
                ctx.push_reads(adm.select((adm.pos < b) & (end > a - 1)))
                res = ctx.finish_contig()
                check_ge(f"L={L} shard [{a},{b})", res, K8, expected(oc, length, L, K8, a, b))
                check_invariants(res)
                parts.append(res)
            vec = sum(pack_counters(p).view(np.uint64) for p in parts)
            whole = unpack_counters(vec.view(np.int64), parts[0])
            check_ge(f"L={L} summed", whole, K8, expected(oc, length, L, K8))
            check_tiles(f"L={L} summed", whole, expected_tiles(oc, length, L))
        ctx.set_depth_tiles(0)
        ctx.set_depth_thresholds(())


# ------------------------------------------------------------------------------------------------ repeated and re-run work
def test_reruns_and_refresh_return_the_same_counts(contexts):
    opt = CallableOptions()
    c = synth.synth_short("chr4", 100_000, seed=79)
    contig = (c.name, 0, c.length, c.ref, c.reads)
    oc = run_oracle([contig], opt, debug=True).contigs[0]
    want = expected(oc, c.length, 1000, K8)
    for ctx in contexts(opt):
        ctx.set_depth_tiles(1000)
        ctx.set_depth_thresholds(K8)
        _, results = assert_parity([contig], opt, ctx)
        _, r1 = ctx.rerun_resident(fetch=True)
        _, r2 = ctx.rerun_resident(fetch=True)
        ctx.rerun_resident(fetch=False)
        r3 = ctx.refresh_counters()
        for what, r in (("finish", results[0]), ("rerun 1", r1), ("rerun 2", r2), ("refresh after rerun 3", r3)):
            check_ge(what, r, K8, want)
        ctx.set_depth_tiles(0)
        ctx.set_depth_thresholds(())


def test_record_capacity_rerun_keeps_the_counts(contexts):
    """REF_N at every other position: more run starts than the first record buffer holds, so clb_finish_contig grows it and
    re-runs the contig from reset accumulators."""
    opt = CallableOptions()
    length = 120_000
    ref = bytearray(H.reference(length, 12))
    ref[1:100_000:2] = b"N" * len(range(1, 100_000, 2))
    c = synth.synth_short("chrR", length, seed=80, depth=12.0)
    run_case(contexts(opt), ("chrR", 0, length, bytes(ref), c.reads), opt, thresholds_list=((1, 4, 8, 12, 16),), ls=(256, 1000))


# ------------------------------------------------------------------------------------------------ switching and errors
def test_switching_thresholds_and_turning_them_off(contexts):
    opt = CallableOptions()
    c = synth.synth_short("chr5", 60_000, seed=81)
    contig = (c.name, 0, c.length, c.ref, c.reads)
    oc = run_oracle([contig], opt, debug=True).contigs[0]
    for ctx in contexts(opt):
        ctx.set_depth_tiles(5000)
        _, off = assert_parity([contig], opt, ctx)
        n_off = ctx.counters_device()[1]
        assert off[0].tile_thresholds is None and off[0].tile_raw_ge is None and off[0].tile_qc_ge is None
        for ths in ((30,), (1, 2**32 - 1), K8):
            ctx.set_depth_thresholds(ths)
            _, on = assert_parity([contig], opt, ctx)
            check_ge(f"T={ths}", on[0], ths, expected(oc, c.length, 5000, ths))
            for f in ("tile_territory", "tile_callable", "tile_raw_sum", "tile_qc_sum", "bins", "intervals"):
                assert np.array_equal(getattr(on[0], f), getattr(off[0], f)), f
        ctx.set_depth_thresholds([])
        _, off2 = assert_parity([contig], opt, ctx)
        assert off2[0].tile_thresholds is None and ctx.counters_device()[1] == n_off
        _, rr = ctx.rerun_resident(fetch=True)
        assert rr.tile_raw_ge is None
        ctx.set_depth_tiles(0)


def test_invalid_settings_are_refused(contexts):
    opt = CallableOptions()
    ctx = contexts(opt)[0]
    for bad in ((0,), (0, 5), (5, 5), (10, 5), tuple(range(1, 10)), (-1,), (2**32,)):
        with pytest.raises(ClbError) as e:
            ctx.set_depth_thresholds(bad)
        assert e.value.code == -1, bad
    c = synth.synth_short("chr6", 20_000, seed=82)
    reads = compact_reads(c.reads, admit_reads(c.reads, opt.pileup_max_depth, 0))
    ctx.set_depth_tiles(0)
    ctx.set_depth_thresholds((10,))                                     # thresholds without tiles
    with pytest.raises(ClbError) as e:
        ctx.begin_contig(0, c.name, c.length, c.ref, c.length)
    assert e.value.code == -1 and "clb_set_depth_thresholds" in str(e.value) and "clb_set_depth_tiles" in str(e.value)
    ctx.set_depth_tiles(1000)
    ctx.begin_contig(0, c.name, c.length, c.ref, c.length)
    with pytest.raises(ClbError) as e:
        ctx.set_depth_thresholds((20,))                                 # while a contig is open
    assert e.value.code == -1
    ctx.push_reads(reads)
    res = ctx.finish_contig()
    assert res.tile_thresholds.tolist() == [10]
    ctx.set_depth_thresholds(())
    ctx.set_depth_tiles(0)


# ------------------------------------------------------------------------------------------------ coverage command
def _cli(cwd, args):
    return subprocess.run([CLI, "coverage", *args], cwd=cwd, capture_output=True, text=True, timeout=600)


def test_cli_threshold_columns(tmp_path):
    cs = [synth.synth_short("chr1", 120_000, seed=41), synth.synth_short("chr2", 60_000, seed=42),
          synth.synth_short("chrM", 16_569, seed=43, depth=300.0)]
    contigs = [(c.name, tid, c.length, c.ref, c.reads) for tid, c in enumerate(cs)]
    bam = str(tmp_path / "in.bam"); fa = str(tmp_path / "ref.fa")
    bamio.write_bam(bam, [(n, l, r) for n, _, l, _, r in contigs])
    bamio.write_fasta(fa, [(n, ref) for n, _, _, ref, _ in contigs])
    ths = (1, 10, 20, 30, 255, 256)
    base = [bam, "-r", fa, "-o", "out.bed", "--depth-tiles", "tiles.tsv", "--depth-tile-size", "2000"]
    (tmp_path / "plain").mkdir(); (tmp_path / "th").mkdir()
    plain = _cli(tmp_path / "plain", base)
    on = _cli(tmp_path / "th", base + ["--depth-thresholds", ",".join(map(str, ths))])
    assert plain.returncode == 0 and on.returncode == 0, (plain.stderr, on.stderr)
    ocs = run_oracle(contigs, CallableOptions(), debug=True).contigs
    assert (tmp_path / "plain" / "tiles.tsv").read_text() == expected_tsv(ocs, 2000)      # byte-identical without the flag
    for f in ("out.bed", "summary.json"):
        assert (tmp_path / "plain" / f).read_bytes() == (tmp_path / "th" / f).read_bytes(), f
    lines = (tmp_path / "th" / "tiles.tsv").read_text().splitlines()
    header = "#contig\tstart\tend\tterritory\tcallable\tmean_raw\tmean_qc\t" + "\t".join(
        [f"raw_ge_{t}" for t in ths] + [f"qc_ge_{t}" for t in ths])
    assert lines[0] == header
    want_rows = []
    plain_lines = expected_tsv(ocs, 2000).splitlines()[1:]
    row = 0
    for oc in ocs:
        raw, qc = expected(oc, oc.length, 2000, ths)
        for t in range(raw.shape[1]):
            want_rows.append(plain_lines[row] + "\t" + "\t".join(str(int(v)) for v in list(raw[:, t]) + list(qc[:, t])))
            row += 1
    assert lines[1:] == want_rows


def test_cli_refuses_bad_threshold_lists(tmp_path):
    c = synth.synth_short("chr1", 30_000, seed=44)
    bam = str(tmp_path / "in.bam"); fa = str(tmp_path / "ref.fa")
    bamio.write_bam(bam, [(c.name, c.length, c.reads)]); bamio.write_fasta(fa, [(c.name, c.ref)])
    base = [bam, "-r", fa, "-o", "out.bed", "--depth-tiles", "t.tsv"]
    for bad in ("", "10,", ",10", "10,,20", "a", "1.5", "-3", "0", "0,10", "20,10", "10,10", "1,2,3,4,5,6,7,8,9", "4294967296",
                "99999999999999999999", " 10"):
        p = _cli(tmp_path, base + ["--depth-thresholds", bad])
        assert p.returncode == 2 and "--depth-thresholds" in p.stderr, bad
    p = _cli(tmp_path, [bam, "-r", fa, "-o", "out.bed", "--depth-thresholds", "10,20"])   # without --depth-tiles
    assert p.returncode == 2 and "--depth-thresholds" in p.stderr
    p = _cli(tmp_path, base + ["--depth-thresholds", "1,2,3,4,5,6,7,4294967295"])
    assert p.returncode == 0, p.stderr[-2000:]
