"""Inputs that sit on either side of every rule that decides which pileup kernel takes a window, and a host model of
those rules.

A window is taken by k_pileup_fast unless k_window_ranges routes it to k_pileup_general up front (shard-first window,
more than 16384 candidates, CIGAR density, the sampled depth proof, no sub-batch size that fits the stage) or the fast
kernel hands it over in flight (a read fails the per-read depth proof, has more than 64 CIGAR ops, or the window holds
more than 96 second-and-later M-segments).  `plan_windows` restates those rules on the host so that the tests can say
which kernel a case was written for, and the CPU tests can check that the generators really land where they should.
Every generator is deterministic.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import List, Optional, Sequence, Tuple

import numpy as np

from decodingustools_b200.soa import ReadColumns, encode_cigar

# kernel constants (clb_kernels.cuh / clb_fast.cuh); the GPU tests check WREAL against clb_window_positions()
WN = 2048                    # window entries of the general kernel (entry 0 is the halo position)
WREAL = WN - 1               # positions per window
F_LOOKBACK = 254             # depth proof: pos[i] - pos[i - 254] >= max span  =>  at most 254 reads over any position
F_XCAP = 96                  # second-and-later M-segments per fast window
F_MAXOPS = 64                # longest CIGAR the fast kernel walks
N_CAND_FAST = 16384          # more candidates: general kernel
F_WSTAGE = 4880              # quality bytes one warp of the fast kernel stages per sub-batch
PACKED_LQ_READS = 4 * 7 * 32  # general kernel: packed-u8 low-BQ counters up to this many candidates (KLQ * BPA * 32), else u32
DEEP_CAND = 65535            # more candidates: k_pileup_classify_deep (32-bit depth fields)
NFIRST = 128                 # general kernel: low-MAPQ thresholds of depths below this come from shared memory

_M_OPS = (0, 7, 8)
_REF_OPS = (0, 2, 3, 7, 8)
_QRY_OPS = (0, 1, 4, 7, 8)


# ------------------------------------------------------------------------------------------------ column building
def columns(pos: Sequence[int], cigars: Sequence[str], mapq, quals: Sequence[np.ndarray], flag=None) -> ReadColumns:
    """Read columns from per-read CIGAR strings and quality arrays (vectorised enough for ~10^5 reads)."""
    n = len(pos)
    ops = [encode_cigar(c) for c in cigars]
    coff = np.zeros(n + 1, np.uint32); coff[1:] = np.cumsum([len(o) for o in ops])
    qoff = np.zeros(n + 1, np.uint64); qoff[1:] = np.cumsum([len(q) for q in quals])
    mq = np.broadcast_to(np.asarray(mapq, np.uint8), (n,))
    fl = np.zeros(n, np.uint16) if flag is None else np.asarray(flag, np.uint16)
    return ReadColumns(np.asarray(pos, np.int32), fl, mq, coff, np.concatenate(ops) if n else np.zeros(0, np.uint32),
                       qoff, np.concatenate(quals).astype(np.uint8) if n else np.zeros(0, np.uint8), np.arange(n, dtype=np.uint32))


def query_len(cigar: str) -> int:
    return int(sum(int(v) >> 4 for v in encode_cigar(cigar) if (int(v) & 15) in _QRY_OPS))


def rotating_quals(lengths: Sequence[int], step: int = 37, start: int = 0) -> List[np.ndarray]:
    """Read i gets bytes (start + step * i + j) mod 256: every value 0..255 appears, in every byte lane."""
    return [((start + step * i + np.arange(l)) % 256).astype(np.uint8) for i, l in enumerate(lengths)]


def reference(length: int, seed: int, n_runs: Sequence[Tuple[int, int]] = ()) -> bytes:
    rng = np.random.default_rng(seed)
    ref = rng.choice(np.frombuffer(b"ACGT", np.uint8), size=length)
    for a, b in n_runs:
        ref[max(a, 0):min(b, length)] = ord("N")
    return ref.tobytes()


# ------------------------------------------------------------------------------------------------ host model of the routing
@dataclass
class WindowPlan:
    w: int
    r_lo: int
    r_hi: int
    n_cand: int
    n_ops: int
    sampled_deep: bool          # k_window_ranges' sampled depth proof fails (indices r_lo + 254 k)
    read_deep: bool             # the fast kernel's per-read depth proof fails for some candidate
    max_ops: int                # longest CIGAR among the live candidates
    x_segments: int             # second-and-later M-segments inside the window (fast kernel layout)
    G: int                      # reads per fast sub-batch chosen by k_window_ranges (0: general)
    shrunk: bool                # the sub-batch size had to be reduced after checking the staged bytes
    reason: Optional[str]       # why the window is general (None: fast)

    @property
    def path(self) -> str:
        if self.reason is None:
            return "fast"
        return "deep" if self.n_cand > DEEP_CAND else "general"


def window_r_lo(pos: np.ndarray, w: int, region_start: int, max_span: int) -> int:
    """First candidate read of window w, as k_window_ranges finds it: pos > halo position - max_span."""
    wb = region_start + w * WREAL - 1
    return int(np.searchsorted(pos.astype(np.int64), wb - max_span + 1, side="left"))


def sample_indices(r_lo: int, r_hi: int) -> range:
    """Reads whose depth proof k_window_ranges samples: r_lo + 254 k, k >= 1."""
    return range(r_lo + F_LOOKBACK, r_hi, F_LOOKBACK)


def _x_segments(reads: ReadColumns, idx: np.ndarray, wb0: int, n_ent: int, min_mapq: int) -> int:
    """Second-and-later M-segments the fast kernel would queue for window entries [0, n_ent) starting at wb0."""
    x = 0
    co, qo = reads.cigar_off.astype(np.int64), reads.qual_off.astype(np.int64)
    for i in idx:
        c0, c1 = co[i], co[i + 1]
        ops = reads.cigar[c0:c1]
        if int(reads.mapq[i]) < min_mapq or (int(reads.flag[i]) & 4) or c1 - c0 > F_MAXOPS:
            continue
        if sum(1 for v in ops if (int(v) & 15) in _M_OPS) < 2:
            continue
        lq = int(qo[i + 1] - qo[i])
        rp, qp, segs = int(reads.pos[i]) - wb0, 0, 0
        for v in ops:
            op, ln = int(v) & 15, int(v) >> 4
            if op in _M_OPS and qp < lq and rp < n_ent:
                l = min(ln, lq - qp)
                if min(rp + l, n_ent) > max(rp, 0):
                    segs += 1
            if op in _REF_OPS and rp < WN:
                rp += ln
            if op in _QRY_OPS:
                qp += ln
        x += max(0, segs - 1)
    return x


def plan_windows(reads: ReadColumns, length: int, region: Optional[Tuple[int, int]] = None, max_span: Optional[int] = None,
                 min_mapq: int = 10, force_general: bool = False) -> List[WindowPlan]:
    """Which kernel takes every window of a contig (reads: the admitted, coordinate-sorted records pushed as one batch)."""
    rs, re_ = region if region is not None else (0, length)
    n_w = (re_ - rs + WREAL - 1) // WREAL
    pos = reads.pos.astype(np.int64)
    if max_span is None:
        max_span = reads.max_ref_span()
    qo = reads.qual_off.astype(np.int64)
    co = reads.cigar_off.astype(np.int64)
    nops = np.diff(co)
    live = ((reads.flag & 4) == 0) & (nops > 0)
    max_qlen = int(np.diff(qo).max()) if reads.n else 0
    long_mode = reads.n_cigar > 4 * reads.n
    plans = []
    for w in range(n_w):
        wb = rs + w * WREAL - 1
        wend = min(wb + WN, re_)
        r_lo = int(np.searchsorted(pos, wb - max_span + 1, side="left"))
        r_hi = int(np.searchsorted(pos, wend, side="left"))
        n = r_hi - r_lo
        q_lo, q_hi = int(qo[r_lo]) & ~15, int(qo[r_hi])
        n_ops = int(co[r_hi] - co[r_lo])
        reason = None
        if force_general or long_mode:
            reason = "all windows"
        elif w == 0 and rs != 0:
            reason = "shard-first"
        elif n > N_CAND_FAST:
            reason = "candidates"
        elif n and n_ops > 8 * n + 64:
            reason = "cigar density"
        sampled = any(pos[i - F_LOOKBACK] + max_span > pos[i] for i in sample_indices(r_lo, r_hi))
        if reason is None and sampled:
            reason = "sampled depth proof"
        G, shrunk = 32, False
        if reason is None and n:
            total = q_hi - q_lo
            if total * 32 > (F_WSTAGE - 16) * n:
                G = ((F_WSTAGE - 16) * n) // total
            ok = G >= 4 and max_qlen != 0 and G * max_qlen + 32 <= F_WSTAGE
            tries = 0
            while tries < 4 and G >= 4 and not ok:
                starts = np.arange(r_lo, r_hi, G)
                ends = np.minimum(starts + G, r_hi)
                staged = ((qo[ends] - (qo[starts] & ~15) + 15) & ~15)
                ok = int(staged.max()) <= F_WSTAGE
                if not ok:
                    G -= max(1, G // 8)
                    shrunk = True
                tries += 1
            if not ok:
                reason = "stage"
        idx = np.arange(r_lo, r_hi)
        big = idx[idx >= F_LOOKBACK]
        read_deep = bool(np.any(pos[big - F_LOOKBACK] + max_span > pos[big])) if big.size else False
        max_ops = int(nops[idx][live[idx]].max()) if n and live[idx].any() else 0
        wb0 = rs + w * WREAL
        xs = _x_segments(reads, idx, wb0, min(WREAL, re_ - wb0), min_mapq)
        if reason is None:
            if read_deep:
                reason = "read depth proof"
            elif max_ops > F_MAXOPS:
                reason = "ops"
            elif xs > F_XCAP:
                reason = "x segments"
        plans.append(WindowPlan(w, r_lo, r_hi, n, n_ops, sampled, read_deep, max_ops, xs, 0 if reason else G, shrunk, reason))
    return plans


def general_count(plans: Sequence[WindowPlan]) -> int:
    return sum(p.reason is not None for p in plans)


# ------------------------------------------------------------------------------------------------ case 1: the depth proof
DEPTH_LEN = 3 * WREAL
PILE_SPAN = 50


def depth_pile(n_pile: int, n_before: int) -> ReadColumns:
    """n_pile reads of 50M at one position of window 1, after n_before reads at one per position and followed by 300
    more.  Depth over the pile position is exactly n_pile, every other position is covered by at most 50 reads, and the
    only read pair closer than the depth proof allows is (first pile read, 255th pile read).  With n_before a multiple
    of 254 that pair is one of the samples of k_window_ranges (r_lo = 0); otherwise only the fast kernel's per-read
    check can see it."""
    b0 = WREAL + 53
    pile_pos = b0 + n_before + PILE_SPAN + 10
    pos = list(range(b0, b0 + n_before)) + [pile_pos] * n_pile + [pile_pos + PILE_SPAN + k for k in range(300)]
    n = len(pos)
    mapq = np.where(np.arange(n) % 7 == 0, 0, 60)
    return columns(pos, ["50M"] * n, mapq, rotating_quals([50] * n, step=11))


def pile_index(n_before: int) -> int:
    """Index of the pile's first read."""
    return n_before


# ------------------------------------------------------------------------------------------------ case 2: quality bytes
QUAL_THRESHOLDS = (0, 1, 2, 20, 127, 128, 129, 254, 255)


def _pad16(cigar: str) -> str:
    """Trailing soft clip so that the read's quality string is a multiple of 16 bytes (keeps every read's first
    quality at phase 0, so a leading clip of a bases puts the segment at phase a)."""
    ql = query_len(cigar)
    pad = -ql % 16
    return cigar + (f"{pad}S" if pad else "")


def quality_shapes() -> List[str]:
    shapes = []
    for a in range(16):                                     # 1 base at every alignment
        shapes.append(_pad16((f"{a}S" if a else "") + "1M"))
    for ln in range(2, 17):                                 # 2..16 bases at every alignment
        for a in range(16):
            shapes.append(_pad16((f"{a}S" if a else "") + f"{ln}M"))
    for ln in (17, 32, 33, 151):
        for a in (0, 1, 8, 15):
            shapes.append(_pad16((f"{a}S" if a else "") + f"{ln}M"))
    for a in (0, 3, 14):                                    # second M-segment: the fast kernel's global X list
        shapes.append(_pad16((f"{a}S" if a else "") + "20M2D30M"))
        shapes.append(_pad16((f"{a}S" if a else "") + "20M3I30M"))
        shapes.append(_pad16((f"{a}S" if a else "") + "7M1D1M1I17M"))
    shapes += ["5S40M19S", "1S60M3S", "13S3M16S"]           # soft clips on both ends
    return shapes


def quality_window(copies: int) -> ReadColumns:
    """Every segment shape of quality_shapes(), `copies` times, one read per position in window 1, qualities rotating
    through 0..255.  copies=1 stays below PACKED_LQ_READS candidates, copies=4 goes above it."""
    shapes = quality_shapes() * copies
    order = np.random.default_rng(7).permutation(len(shapes))
    cigars = [shapes[i] for i in order]
    pos = [WREAL + 13 + i for i in range(len(cigars))]
    mapq = np.where(np.arange(len(cigars)) % 9 == 4, 5, 60)
    return columns(pos, cigars, mapq, rotating_quals([query_len(c) for c in cigars], step=37, start=copies))


def deep_quality_window(n: int = 70_000) -> ReadColumns:
    """More than 65535 short reads (1..33 bases, rotating qualities) in window 1: the deep kernel."""
    rng = np.random.default_rng(5)
    pos = np.sort(rng.integers(WREAL, 2 * WREAL - 40, n))
    lens = rng.integers(1, 34, n)
    ops = (lens.astype(np.uint32) << 4)
    qual = ((np.arange(int(lens.sum())) * 7 + 3) % 256).astype(np.uint8)
    coff = np.arange(n + 1, dtype=np.uint32)
    qoff = np.zeros(n + 1, np.uint64); qoff[1:] = np.cumsum(lens)
    mapq = np.where(np.arange(n) % 5 == 0, 0, 60).astype(np.uint8)
    return ReadColumns(pos.astype(np.int32), np.zeros(n, np.uint16), mapq, coff, ops, qoff, qual, np.arange(n, dtype=np.uint32))


# ------------------------------------------------------------------------------------------------ case 3: threshold tables
FRACTIONS = (0.0, -0.0, 0.1, 0.2, 1 / 3, 0.5, math.nextafter(0.25, 1.0), 0.999999, 1.0, -0.5)
STAIR_SPLIT = 255             # raw depths from here on start a window of their own (a fast window cannot hold them)
STAIR_WINDOW_READS = 16_000   # reads per staircase window (a fast window takes at most 16384 candidates)


def first_low(raw: int, fraction: float) -> int:
    """Smallest low-MAPQ count with low / raw > fraction (callable_profiler.rs:100-101), raw + 1 if there is none."""
    for low in range(raw + 2):
        if low / raw > fraction:
            return low
    return raw + 1


def staircase_steps(fraction: float, max_raw: int = 300) -> List[Tuple[int, int, int, int]]:
    """(position, raw, low, window): for raw 1..max_raw, low at the threshold and one below (clipped to [0, raw]).  Steps
    are two positions apart so that the pileup never holds two steps at once (the admission cap counts live reads); a
    window takes at most STAIR_WINDOW_READS reads, and the depths from 255 on start a new window."""
    steps, w, p, in_w = [], 0, 11, 0
    for raw in range(1, max_raw + 1):
        t = first_low(raw, fraction)
        for low in sorted({min(max(t - 1, 0), raw), min(t, raw)}):
            if in_w + raw > STAIR_WINDOW_READS or (raw == STAIR_SPLIT and in_w and steps[-1][1] < STAIR_SPLIT):
                w += 1; p = w * WREAL + 11; in_w = 0
            steps.append((p, raw, low, w))
            p += 2; in_w += raw
    return steps


def staircase_len(fraction: float, max_raw: int = 300) -> int:
    return (staircase_steps(fraction, max_raw)[-1][3] + 2) * WREAL


def staircase(fraction: float, max_low_mapq: int = 1, high_mapq: int = 60, max_raw: int = 300) -> ReadColumns:
    """Position p holds raw(p) reads of 1M, low(p) of them with MAPQ max_low_mapq and the rest with high_mapq."""
    steps = staircase_steps(fraction, max_raw)
    raw = np.array([s[1] for s in steps]); low = np.array([s[2] for s in steps])
    pos = np.repeat([s[0] for s in steps], raw).astype(np.int32)
    n = pos.shape[0]
    k = np.arange(n) - np.repeat(np.cumsum(raw) - raw, raw)           # index of the read within its step
    mapq = np.where(k < np.repeat(low, raw), max_low_mapq, high_mapq).astype(np.uint8)
    return ReadColumns(pos, np.zeros(n, np.uint16), mapq, np.arange(n + 1, dtype=np.uint32), np.full(n, 16, np.uint32),
                       np.arange(n + 1, dtype=np.uint64), ((np.arange(n) * 13) % 256).astype(np.uint8), np.arange(n, dtype=np.uint32))


# ------------------------------------------------------------------------------------------------ case 4: bail limits
BAIL_LEN = 3 * WREAL


def x_segment_window(n_x: int) -> ReadColumns:
    """n_x reads with a second M-segment (20M2D30M) among 1-op reads, all inside window 1."""
    cigars = ["20M2D30M" if i % 2 == 0 and i // 2 < n_x else "50M" for i in range(2 * n_x + 20)]
    pos = [WREAL + 20 + 3 * i for i in range(len(cigars))]
    return columns(pos, cigars, 60, rotating_quals([50] * len(cigars), step=29))


def ops_window(n_ops: int) -> ReadColumns:
    """One read of n_ops CIGAR ops (64: walked by the fast kernel, 65: handed over) among 30 reads of one op."""
    long = "20M" + "".join("1I" if k % 2 == 0 else "1D" for k in range(62)) + "20M"
    assert len(encode_cigar(long)) == 64
    if n_ops == 65:
        long += "5S"
    cigars = ["60M"] * 15 + [long] + ["60M"] * 15
    pos = [WREAL + 100 + 10 * i for i in range(len(cigars))]
    return columns(pos, cigars, 60, rotating_quals([query_len(c) for c in cigars], step=3))


def candidate_window(n_cand: int) -> ReadColumns:
    """1-base reads at depth 8 over the 2048 entries (halo included) of window 1: 16384 candidates; one more read
    (depth 9 at one position) makes 16385."""
    wb = WREAL - 1
    pos = np.repeat(np.arange(wb, wb + WN), 8)
    extra = n_cand - pos.shape[0]
    assert 0 <= extra <= 8
    pos = np.sort(np.concatenate([pos, np.full(extra, wb + 1000)])).astype(np.int32)
    n = pos.shape[0]
    return ReadColumns(pos, np.zeros(n, np.uint16), np.where(np.arange(n) % 11 == 0, 0, 60).astype(np.uint8),
                       np.arange(n + 1, dtype=np.uint32), np.full(n, 16, np.uint32), np.arange(n + 1, dtype=np.uint64),
                       ((np.arange(n) * 31) % 256).astype(np.uint8), np.arange(n, dtype=np.uint32))


def density_window(extra: int) -> ReadColumns:
    """16 reads in window 1 whose CIGAR ops add up to 8 * 16 + 64 + extra."""
    target = 8 * 16 + 64 + extra
    ks = [(target - 32) // 16] * 16
    ks[-1] += target - 32 - sum(ks)
    cigars = ["10M" + "".join("1I" if j % 2 == 0 else "1D" for j in range(k)) + "10M" for k in ks]
    pos = [WREAL + 200 + 100 * i for i in range(16)]
    # 80 one-op reads in window 0 keep the batch at most 4 ops per read (more would switch the contig to long-read mode)
    cigars = ["10M"] * 80 + cigars
    pos = [100 + 20 * i for i in range(80)] + pos
    return columns(pos, cigars, 60, rotating_quals([query_len(c) for c in cigars], step=5))


STAGE_TOTALS = (4864, 4865, 4879, 4880)
STAGE_PHASES = (0, 1, 8, 15)


def stage_window(total: int, phase: int) -> ReadColumns:
    """Four reads of ~1216 quality bytes (16 aligned bases each, the rest soft-clipped) whose qualities add up to
    `total`, followed by four 10-base reads, in window 1; a read in window 0 puts the first of them at 16-byte phase
    `phase`.  The mean read length makes k_window_ranges start at 7 reads per sub-batch and shrink to 4, where the
    four long reads stage p + total bytes rounded up to 16: they fit the 4880-byte stage iff phase + total <= 4880;
    otherwise the next step (3 reads) is below the fast kernel's minimum and the window goes to the general kernel."""
    lens = [total // 4] * 4
    lens[-1] += total - sum(lens)
    cigars = [f"{16 + phase}M"] + [f"16M{l - 16}S" for l in lens] + ["10M"] * 4
    pos = [10] + [3000 + i for i in range(8)]
    return columns(pos, cigars, 60, rotating_quals([query_len(c) for c in cigars], step=17))


def mixed_lengths(seed: int = 3, length: int = 4 * WREAL) -> ReadColumns:
    """Reads of 36..400 bases at random positions (~25x): no single sub-batch size suits every window, so the uniform
    max-length shortcut of k_window_ranges fails and its shrink loop sizes the sub-batches."""
    rng = np.random.default_rng(seed)
    lens = rng.choice([36, 75, 151, 250, 400], size=1200, p=[.3, .2, .2, .2, .1])
    pos = np.sort(rng.integers(0, length - 400, lens.shape[0]))
    cigars = [f"{l}M" if i % 5 else f"{l // 2}M3D{l - l // 2}M" for i, l in enumerate(lens)]
    mapq = rng.choice([0, 5, 60], size=lens.shape[0], p=[.1, .1, .8])
    return columns(pos, cigars, mapq, rotating_quals(lens, step=23))


# ------------------------------------------------------------------------------------------------ case 5: seams
SEAM_WINDOWS = 8
SEAM_LEN = SEAM_WINDOWS * WREAL
SEAM_PILES = (2, 3, 5)        # windows with a 300-read pile: fast, fast, general, general, fast, general, fast, fast
SEAM_FEATURES = ("continue", "n_through", "n_ends", "n_starts", "gap_through", "gap_ends", "gap_starts", "depth_step")


def seam_contig(feature: str, seed: int = 41) -> Tuple[bytes, ReadColumns]:
    """An 8-window contig at ~12x (100M reads) with a 300-read pile in the middle of windows 2, 3 and 5, and one kind of
    state change (or none) placed exactly at every window seam s = w * WREAL."""
    rng = np.random.default_rng(seed)
    seams = [w * WREAL for w in range(1, SEAM_WINDOWS)]
    n_runs = []
    if feature == "n_through":
        n_runs = [(s - 6, s + 6) for s in seams]
    elif feature == "n_ends":
        n_runs = [(s - 9, s) for s in seams]
    elif feature == "n_starts":
        n_runs = [(s, s + 9) for s in seams]
    ref = reference(SEAM_LEN, seed, n_runs)
    starts = np.sort(rng.integers(0, SEAM_LEN - 100, int(12 * SEAM_LEN / 100)))
    keep = np.ones(starts.shape[0], bool)
    for s in seams:
        if feature == "gap_through":
            keep &= ~((starts < s + 20) & (starts + 100 > s - 20))
        elif feature == "gap_ends":
            keep &= ~((starts < s) & (starts + 100 > s - 20))
        elif feature == "gap_starts":
            keep &= ~((starts < s + 20) & (starts + 100 > s))
    starts = list(starts[keep])
    mapq = list(rng.choice([60, 60, 60, 30, 0], size=len(starts)))
    for s in seams:
        if feature == "gap_ends":
            starts += [s] * 6; mapq += [60] * 6                       # coverage resumes exactly at the seam
        elif feature == "gap_starts":
            starts += [s - 100] * 6; mapq += [60] * 6                 # ... and stops exactly at it
        elif feature == "depth_step":
            starts += [s - 100] * 80; mapq += [60] * 80               # 80 more reads end at the seam
            starts += [s] * 40; mapq += [0] * 40                      # 40 MAPQ-0 reads start at it: POOR_MAPPING_QUALITY
    for w in SEAM_PILES:
        starts += [w * WREAL + 1000] * 300; mapq += [60] * 300
    order = np.argsort(np.array(starts), kind="stable")
    pos = [int(starts[i]) for i in order]
    mq = np.array([mapq[i] for i in order], np.uint8)
    return ref, columns(pos, ["100M"] * len(pos), mq, rotating_quals([100] * len(pos), step=19))


# ------------------------------------------------------------------------------------------------ case 6: synthetic contigs
SYNTH_CASES = ((36, 60.0), (75, 30.0), (100, 15.0), (151, 45.0), (250, 30.0), (150, 230.0), (150, 300.0))
SYNTH_LEN = 300_000
