"""Region sharding across GPUs (SURVEY.md section 8(e); BASELINE.json north_star "partitioned ... by contig and
fixed-size genomic region, with halo reads at region boundaries and interval stitching on the host").

Columns of the pileup are independent once the admitted read set is fixed, so a contig is cut into contiguous
regions (one per rank), each rank receives every admitted read that overlaps its region or the single base to its
left (the halo that lets the kernel decide whether the region's first run continues the previous one), and the
only exchange is a sum of the additive counters + bins (NCCL all-reduce on the GPU box, gloo in the CPU tests) plus
a host-side concatenation of the per-region interval lists.  The reference is single-process and single-threaded
(/root/reference/src/api/coverage.rs:221-236); nothing here has a counterpart there.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Sequence, Tuple

import numpy as np

from .callable_loci import INTERVAL_DTYPE, RUN_DTYPE, ContigDeviceResult, stitch_depth_runs, stitch_intervals
from .soa import ReadColumns


@dataclass(frozen=True)
class Shard:
    tid: int
    start: int
    end: int


def plan_regions(contig_lengths: Sequence[int], world_size: int, window: int) -> List[List[Shard]]:
    """Cut the genome (contigs in tid order) into `world_size` runs of roughly equal size; cuts inside a contig fall
    on multiples of the kernel's window size so no window is split between ranks.  Returns shards per rank."""
    total = int(sum(contig_lengths))
    per_rank: List[List[Shard]] = [[] for _ in range(world_size)]
    if total == 0:
        return per_rank
    target = total / world_size
    rank, used = 0, 0.0
    for tid, length in enumerate(contig_lengths):
        pos = 0
        while pos < length:
            room = target * (rank + 1) - used
            if rank == world_size - 1 or room >= length - pos:
                take = length - pos
            else:
                take = int(round(room / window)) * window
                take = max(window, take) if room > 0 else 0
                take = min(take, length - pos)
            if take > 0:
                mine = per_rank[rank]
                if mine and mine[-1].tid == tid and mine[-1].end == pos:
                    mine[-1] = Shard(tid, mine[-1].start, pos + take)     # contiguous with the rank's previous piece: one shard
                else:
                    mine.append(Shard(tid, pos, pos + take))
                pos += take; used += take
            if used >= target * (rank + 1) - 1e-9 and rank < world_size - 1:
                rank += 1
    return per_rank


def reads_for_region(reads: ReadColumns, start: int, end: int, max_ref_span: int | None = None) -> Tuple[int, int]:
    """Record range [lo, hi) that contains every read overlapping [start - 1, end) (coordinate-sorted columns)."""
    if reads.n == 0:
        return 0, 0
    span = reads.max_ref_span() if max_ref_span is None else int(max_ref_span)
    lo = int(np.searchsorted(reads.pos, start - 1 - span + 1, side="left"))
    hi = int(np.searchsorted(reads.pos, end, side="left"))
    return lo, max(lo, hi)


COUNTER_FIELDS = ("n_covered_bases", "summed_coverage", "summed_baseq", "summed_mapq", "quality_bases")
TILE_FIELDS = ("tile_territory", "tile_callable", "tile_raw_sum", "tile_qc_sum")


def pack_counters(res: ContigDeviceResult) -> np.ndarray:
    """The additive part of a shard result as one int64 vector: 6 state counts, 5 sums, 3 * n_bins bins, then the raw and
    QC depth histograms when they are on, then the tiles' territory, callable, raw_sum and qc_sum when they are on (the
    order of the device's counter buffer)."""
    head = np.array(list(res.state_counts) + [getattr(res, k) for k in COUNTER_FIELDS], dtype=np.uint64)
    parts = [head, res.bins.astype(np.uint64).ravel()]
    if res.depth_hist_raw is not None:
        parts += [np.asarray(res.depth_hist_raw, np.uint64), np.asarray(res.depth_hist_qc, np.uint64)]
    if res.tile_territory is not None:
        parts += [np.asarray(getattr(res, k), np.uint64) for k in TILE_FIELDS]
    return np.concatenate(parts).view(np.int64)


def unpack_counters(vec: np.ndarray, res: ContigDeviceResult) -> ContigDeviceResult:
    """Inverse of pack_counters; whether `res` has depth histograms and tiles (and their lengths) says how the tail splits."""
    v = np.asarray(vec).view(np.uint64)
    res.state_counts = v[:6].copy()
    for i, k in enumerate(COUNTER_FIELDS):
        setattr(res, k, int(v[6 + i]))
    n = 0 if res.depth_hist_raw is None else len(res.depth_hist_raw)
    nt = 0 if res.tile_territory is None else len(res.tile_territory)
    end = v.shape[0] - 2 * n - 4 * nt
    res.bins = v[11:end].reshape(3, -1).astype(np.uint32)
    if n:
        res.depth_hist_raw = v[end:end + n].copy()
        res.depth_hist_qc = v[end + n:end + 2 * n].copy()
    for i, k in enumerate(TILE_FIELDS if nt else ()):
        setattr(res, k, v[end + 2 * n + i * nt:end + 2 * n + (i + 1) * nt].copy())
    return res


def allreduce_counters(res: ContigDeviceResult, group=None) -> ContigDeviceResult:
    """Sum the additive counters of one contig over all ranks (integer sums: order independent, bit exact)."""
    import torch
    import torch.distributed as dist
    t = torch.from_numpy(pack_counters(res).copy())
    if dist.get_backend(group) == "nccl":
        t = t.cuda()
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return unpack_counters(t.cpu().numpy(), res)


def _gather_sorted(local: np.ndarray, dtype: np.dtype, region_start: int, dst: int, group):
    """The per-rank arrays of one contig on `dst`, in genomic order (None elsewhere)."""
    import torch.distributed as dist
    payload = (int(region_start), np.ascontiguousarray(local, dtype=dtype).tobytes())
    gathered = [None] * dist.get_world_size(group) if dist.get_rank(group) == dst else None
    dist.gather_object(payload, gathered, dst=dst, group=group)
    if gathered is None:
        return None
    return [np.frombuffer(b, dtype=dtype) for _, b in sorted((p for p in gathered if len(p[1])), key=lambda p: p[0])]


def gather_and_stitch(local_intervals: np.ndarray, region_start: int, dst: int = 0, group=None):
    """Collect the per-rank interval lists of one contig on `dst` and stitch them in genomic order."""
    parts = _gather_sorted(local_intervals, INTERVAL_DTYPE, region_start, dst, group)
    return None if parts is None else stitch_intervals(parts)


def gather_and_stitch_depth_runs(local_runs: np.ndarray, region_start: int, dst: int = 0, group=None):
    """Same for the depth runs (ContigDeviceResult.depth_runs): they are not additive, so they are gathered, not summed."""
    parts = _gather_sorted(local_runs, RUN_DTYPE, region_start, dst, group)
    return None if parts is None else stitch_depth_runs(parts)
