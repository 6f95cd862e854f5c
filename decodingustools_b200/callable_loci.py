"""Host-side mirror of the reference's `callable_loci` module over the C-ABI device library.

Names follow the reference so the tests read like tests of the original:
    process_single_contig   /root/reference/src/callable_loci/mod.rs:44-147
    CallableProfiler        /root/reference/src/callable_loci/profilers/callable_profiler.rs
    ContigProfiler          /root/reference/src/callable_loci/profilers/contig_profiler.rs

The per-base work (pileup, classification, run-length segmentation, sums, bins) happens on the GPU
inside :class:`CallableLociContext`; this module keeps what the north_star leaves on the host: read
admission (htslib's depth cap), unique read-name counting, the BED text with the reference's
cross-contig behaviour, and the final floating-point aggregation (report.py).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from ._lib import ClbError
from .options import CallableOptions
from .soa import ReadColumns

INTERVAL_DTYPE = np.dtype([("start", "<u4"), ("end", "<u4"), ("state", "u1"), ("soft_start", "u1"), ("_pad", "<u2")])
assert INTERVAL_DTYPE.itemsize == C.sizeof(_lib.Interval) == 12
# clb_depth_run: a run of equal raw or QC depth starts at `start` and ends where the next one starts (the last: at the region
# end)
RUN_DTYPE = np.dtype([("start", "<u4"), ("depth", "<u4")])


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _c_options(o: CallableOptions) -> _lib.Options:
    return _lib.Options(o.min_depth, o.max_depth, o.min_depth_for_low_mapq, o.min_mapping_quality,
                        o.min_base_quality, o.max_low_mapq, 0, float(o.max_low_mapq_fraction))


@dataclass
class ContigDeviceResult:
    """What the device computes for one contig or region shard (clb_contig_result)."""
    state_counts: np.ndarray
    n_covered_bases: int
    summed_coverage: int
    summed_baseq: int
    summed_mapq: int
    quality_bases: int
    intervals: np.ndarray          # INTERVAL_DTYPE
    bins: np.ndarray               # uint32[3, n_bins]
    stride: int
    region_start: int
    region_end: int
    kernel_ms: float = 0.0
    h2d_ms: float = 0.0
    pileup_ms: float = 0.0
    h2d_bytes: int = 0
    d2h_bytes: int = 0
    gpu_launches: int = 0
    fast_ms: float = 0.0
    general_windows: int = 0
    upload_ms: float = 0.0
    # depth histograms (set_depth_histogram): uint64[n] each, None when off.  Bin d counts the positions that are not REF_N
    # with raw / QC depth d; the last bin counts every depth >= n - 1.
    depth_hist_raw: Optional[np.ndarray] = None
    depth_hist_qc: Optional[np.ndarray] = None
    # depth tiles (set_depth_tiles): uint64[n_tiles] each, None when off.  Tile t covers contig positions
    # [t * tile_len, min((t + 1) * tile_len, length)); territory counts its positions that are not REF_N, callable the
    # CALLABLE ones, raw_sum / qc_sum the raw / QC depth summed over the territory (mean depth: sum / territory).
    tile_len: int = 0
    tile_territory: Optional[np.ndarray] = None
    tile_callable: Optional[np.ndarray] = None
    tile_raw_sum: Optional[np.ndarray] = None
    tile_qc_sum: Optional[np.ndarray] = None
    # depth thresholds per tile (set_depth_thresholds, with the tiles): the thresholds, uint32[K], and per threshold j and
    # tile t the tile's positions that are not REF_N with raw / QC depth >= tile_thresholds[j], uint64[K, n_tiles] each;
    # None when off.
    tile_thresholds: Optional[np.ndarray] = None
    tile_raw_ge: Optional[np.ndarray] = None
    tile_qc_ge: Optional[np.ndarray] = None
    # depth runs (set_depth_runs): RUN_DTYPE[n], None when off.  The raw depth of every position of the region as runs of
    # equal depth (depth_run_ends gives their ends); region shards join with stitch_depth_runs.
    depth_runs: Optional[np.ndarray] = None
    # QC depth runs (set_qc_depth_runs): the same for the QC depth, the depth the states are called on (the depth behind
    # quality_bases); RUN_DTYPE[n], None when off.
    qc_depth_runs: Optional[np.ndarray] = None


def _result(res: _lib.ContigResult, copy_intervals: bool = True) -> ContigDeviceResult:
    n = int(res.n_intervals)
    if n and copy_intervals:
        iv = np.ctypeslib.as_array(C.cast(res.intervals, C.POINTER(C.c_uint8)), shape=(n * 12,)).view(INTERVAL_DTYPE).copy()
    else:
        iv = np.zeros(0, dtype=INTERVAL_DTYPE)
    nb = int(res.n_bins)
    bins = np.ctypeslib.as_array(res.bins, shape=(3 * nb,)).reshape(3, nb).copy() if nb else np.zeros((3, 0), np.uint32)
    return ContigDeviceResult(np.array(list(res.state_counts), dtype=np.uint64), int(res.n_covered_bases),
                              int(res.summed_coverage), int(res.summed_baseq), int(res.summed_mapq), int(res.quality_bases),
                              iv, bins, int(res.stride), int(res.region_start), int(res.region_end), float(res.kernel_ms),
                              float(res.h2d_ms), float(res.pileup_ms), int(res.h2d_bytes), int(res.d2h_bytes), int(res.gpu_launches),
                              float(res.fast_ms), int(res.general_windows), float(res.upload_ms))


def depth_run_ends(runs: np.ndarray, region_end: int) -> np.ndarray:
    """End of each depth run (raw or QC): the next run's start, region_end for the last."""
    starts = np.asarray(runs["start"], dtype=np.int64)
    return np.append(starts[1:], np.int64(region_end)) if starts.size else np.zeros(0, np.int64)


def stitch_depth_runs(shards: Sequence[np.ndarray]) -> np.ndarray:
    """Concatenate the depth runs (raw or QC) of region shards of one contig in genomic order, dropping a shard's first run
    when its depth equals the previous shard's last (runs are defined by depth alone)."""
    parts: List[np.ndarray] = []
    last = None
    for s in shards:
        s = np.ascontiguousarray(s, dtype=RUN_DTYPE)
        if s.size and last is not None and s["depth"][0] == last:
            s = s[1:]
        if s.size:
            parts.append(s)
            last = s["depth"][-1]
    return np.concatenate(parts) if parts else np.zeros(0, RUN_DTYPE)


def depth_tile_ranges(length: int, tile_len: int) -> Tuple[np.ndarray, np.ndarray]:
    """(start, end) of the depth tiles of a contig of `length` positions (set_depth_tiles): tile t covers
    [t * tile_len, min((t + 1) * tile_len, length)), so the last tile may be partial and a tile longer than the contig is
    one tile covering all of it."""
    n = -(-int(length) // int(tile_len))
    start = np.arange(n, dtype=np.int64) * int(tile_len)
    return start, np.minimum(start + int(tile_len), int(length))


class CallableLociContext:
    """One device context (one per GPU / process).  Not thread-safe, like the reference's profilers."""

    def __init__(self, options: CallableOptions, device: int = 0):
        self._L = _lib.lib()
        self.options = options
        err = C.create_string_buffer(512)
        co = _c_options(options)
        self._h = self._L.clb_create(int(device), C.byref(co), err, 512)
        if not self._h:
            raise ClbError(-2, err.value.decode() or "clb_create failed")
        self._keep: list = []

    def close(self):
        if getattr(self, "_h", None):
            self._L.clb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _check(self, rc: int):
        if rc != 0:
            raise ClbError(rc, self._L.clb_last_error(self._h).decode())

    def set_depth_histogram(self, n_bins: int):
        """Raw- and QC-depth histograms of n_bins bins (2..65536; 0: off, the default) from the next begin_contig on."""
        self._check(self._L.clb_set_depth_histogram(self._h, int(n_bins)))

    def set_depth_tiles(self, tile_len: int):
        """Per-tile territory, callable count and raw / QC depth sums over tiles of tile_len positions (256..2^31; 0: off,
        the default) from the next begin_contig on."""
        self._check(self._L.clb_set_depth_tiles(self._h, int(tile_len)))

    def set_depth_thresholds(self, thresholds: Sequence[int]):
        """Per depth tile, the positions with raw / QC depth >= each of 1..8 strictly ascending thresholds (1..2^32-1; an
        empty sequence: off, the default) from the next begin_contig on.  Needs depth tiles on (set_depth_tiles)."""
        vals = [int(t) for t in thresholds]
        if any(t < 0 or t > 0xffffffff for t in vals):
            raise ClbError(-1, f"depth thresholds {vals}: each 1..2^32-1")
        arr = (C.c_uint32 * max(len(vals), 1))(*vals)
        self._check(self._L.clb_set_depth_thresholds(self._h, arr, len(vals)))

    def set_depth_runs(self, on: bool):
        """Runs of equal raw depth over every position of the region (off by default) from the next begin_contig on."""
        self._check(self._L.clb_set_depth_runs(self._h, 1 if on else 0))

    def set_qc_depth_runs(self, on: bool):
        """Runs of equal QC depth over every position of the region (off by default) from the next begin_contig on;
        independent of set_depth_runs."""
        self._check(self._L.clb_set_qc_depth_runs(self._h, 1 if on else 0))

    def _with_optional_counts(self, r: ContigDeviceResult) -> ContigDeviceResult:
        raw = C.POINTER(C.c_uint64)(); qc = C.POINTER(C.c_uint64)(); n = C.c_uint32(0)
        self._check(self._L.clb_depth_histogram(self._h, C.byref(raw), C.byref(qc), C.byref(n)))
        if n.value:
            r.depth_hist_raw = np.ctypeslib.as_array(raw, shape=(n.value,)).copy()
            r.depth_hist_qc = np.ctypeslib.as_array(qc, shape=(n.value,)).copy()
        arrs = [C.POINTER(C.c_uint64)() for _ in range(4)]; nt = C.c_uint32(0); tl = C.c_uint32(0)
        self._check(self._L.clb_depth_tiles(self._h, *[C.byref(a) for a in arrs], C.byref(nt), C.byref(tl)))
        if nt.value:
            r.tile_len = int(tl.value)
            r.tile_territory, r.tile_callable, r.tile_raw_sum, r.tile_qc_sum = (
                np.ctypeslib.as_array(a, shape=(nt.value,)).copy() for a in arrs)
        rg = C.POINTER(C.c_uint64)(); qg = C.POINTER(C.c_uint64)(); th = C.POINTER(C.c_uint32)(); k = C.c_uint32(0)
        self._check(self._L.clb_depth_tile_thresholds(self._h, C.byref(rg), C.byref(qg), C.byref(th), C.byref(k), C.byref(nt)))
        if k.value:
            shape = (k.value, nt.value)
            r.tile_thresholds = np.ctypeslib.as_array(th, shape=(k.value,)).copy()
            r.tile_raw_ge = np.ctypeslib.as_array(rg, shape=shape).copy()
            r.tile_qc_ge = np.ctypeslib.as_array(qg, shape=shape).copy()
        for fn, field in ((self._L.clb_depth_runs, "depth_runs"), (self._L.clb_qc_depth_runs, "qc_depth_runs")):
            rp = C.c_void_p(0); nr = C.c_uint64(0)
            self._check(fn(self._h, C.byref(rp), C.byref(nr)))
            if rp.value:
                n = int(nr.value)
                setattr(r, field, np.ctypeslib.as_array(C.cast(rp, C.POINTER(C.c_uint8)), shape=(n * 8,)).view(RUN_DTYPE).copy()
                        if n else np.zeros(0, RUN_DTYPE))
        return r

    def set_stream(self, cuda_stream: int):
        self._check(self._L.clb_set_stream(self._h, C.c_void_p(int(cuda_stream) or None)))

    def begin_contig(self, tid: int, name: str, length: int, ref, largest_contig_len: int,
                     region: Optional[Tuple[int, int]] = None, max_ref_span: int = 0, ref_is_nmask: bool = False):
        if ref is None:
            ref_arr, ref_len = None, 0
        elif ref_is_nmask:
            ref_arr = np.ascontiguousarray(ref, dtype=np.uint32); ref_len = ref_arr.shape[0]
        else:
            ref_arr = np.frombuffer(ref, dtype=np.uint8) if isinstance(ref, (bytes, bytearray)) else np.ascontiguousarray(ref, dtype=np.uint8)
            ref_len = ref_arr.shape[0]
        r0, r1 = region if region is not None else (0, length)
        self._keep = [ref_arr]
        self._check(self._L.clb_begin_contig(self._h, int(tid), name.encode(), int(length), _ptr(ref_arr), int(ref_len),
                                             1 if ref_is_nmask else 0, int(largest_contig_len), int(r0), int(r1), int(max_ref_span)))

    def reserve(self, n_reads: int, n_cigar: int, n_qual: int):
        self._check(self._L.clb_reserve(self._h, int(n_reads), int(n_cigar), int(n_qual)))

    def push_reads(self, rc: ReadColumns):
        """Append an admitted, coordinate-sorted column batch (offsets relative to the batch)."""
        if rc.n == 0:
            return
        b = _lib.ReadBatch(rc.n, rc.n_cigar, rc.n_qual, _ptr(rc.pos), _ptr(rc.flag), _ptr(rc.mapq), _ptr(rc.cigar_off),
                           _ptr(rc.cigar), _ptr(rc.qual_off), _ptr(rc.qual))
        self._keep.append(rc)          # async copies read these buffers until finish_contig
        self._check(self._L.clb_push_reads(self._h, C.byref(b)))

    def push_raw(self, n_reads, n_cigar, n_qual, pos, flag, mapq, cigar_off, cigar, qual_off, qual):
        """Same as push_reads but from raw addresses (e.g. pinned torch tensors' data_ptr())."""
        b = _lib.ReadBatch(int(n_reads), int(n_cigar), int(n_qual), pos, flag, mapq, cigar_off, cigar, qual_off, qual)
        self._check(self._L.clb_push_reads(self._h, C.byref(b)))

    def finish_contig(self, copy_intervals: bool = True) -> ContigDeviceResult:
        res = _lib.ContigResult()
        self._check(self._L.clb_finish_contig(self._h, C.byref(res)))
        self._keep = self._keep[:1]
        return self._with_optional_counts(_result(res, copy_intervals))

    def finish_contig_raw(self) -> "_lib.ContigResult":
        """clb_finish_contig without copying anything out: the struct's pointers stay valid until the next begin_contig."""
        res = _lib.ContigResult()
        self._check(self._L.clb_finish_contig(self._h, C.byref(res)))
        self._keep = self._keep[:1]
        return res

    def allreduce_nccl(self, nccl_comm: int):
        """Sum the counter buffer over the ranks of an ncclComm_t (enqueued on the compute stream)."""
        self._check(self._L.clb_allreduce_nccl(self._h, C.c_void_p(int(nccl_comm))))

    def rerun_resident(self, fetch: bool = True, copy_intervals: bool = False, sync: bool = True):
        if not fetch and not sync:                       # enqueue only (clb_rerun_resident(ctx, NULL, NULL))
            self._check(self._L.clb_rerun_resident(self._h, None, None))
            return None, None
        ms = C.c_float(0)
        if fetch:
            res = _lib.ContigResult()
            self._check(self._L.clb_rerun_resident(self._h, C.byref(res), C.byref(ms)))
            return float(ms.value), self._with_optional_counts(_result(res, copy_intervals))
        self._check(self._L.clb_rerun_resident(self._h, None, C.byref(ms)))
        return float(ms.value), None

    def counters_device(self) -> Tuple[int, int]:
        p = C.c_void_p(0); n = C.c_uint64(0)
        self._check(self._L.clb_counters_device(self._h, C.byref(p), C.byref(n)))
        return int(p.value), int(n.value)

    def refresh_counters(self) -> ContigDeviceResult:
        res = _lib.ContigResult()
        self._check(self._L.clb_refresh_counters(self._h, C.byref(res)))
        return self._with_optional_counts(_result(res, True))

    def debug_per_base(self, n: int):
        raw = np.zeros(n, np.uint32); qc = np.zeros(n, np.uint32); low = np.zeros(n, np.uint32); st = np.zeros(n, np.uint8)
        self._check(self._L.clb_debug_per_base(self._h, _ptr(raw), _ptr(qc), _ptr(low), _ptr(st)))
        return raw, qc, low, st


# ------------------------------------------------------------------------------------------------
# Host half
# ------------------------------------------------------------------------------------------------
def admit_reads(reads: ReadColumns, maxcnt: int, tid: int = 0, threads: Optional[int] = None, max_ref_span: int = 0,
                stats: Optional[dict] = None) -> np.ndarray:
    """htslib's pileup admission (depth cap) as the reference configures it: mod.rs:55-60.
    threads=None: the sequential recurrence (clb_admit_reads); otherwise the parallel form (clb_admit_reads_mt, 0 = all cores)."""
    keep = np.zeros(reads.n, dtype=np.uint8)
    if threads is None:
        rc = _lib.lib().clb_admit_reads(int(tid), int(maxcnt), reads.n, _ptr(reads.pos), _ptr(reads.flag), _ptr(reads.cigar_off),
                                        _ptr(reads.cigar), _ptr(keep))
    else:
        n_rep = C.c_uint64(0)
        rc = _lib.lib().clb_admit_reads_mt(int(tid), int(maxcnt), reads.n, _ptr(reads.pos), _ptr(reads.flag), _ptr(reads.cigar_off),
                                           _ptr(reads.cigar), int(max_ref_span), int(threads), _ptr(keep), C.byref(n_rep))
        if stats is not None:
            stats["replayed"] = int(n_rep.value)
    if rc != 0:
        raise ClbError(rc, "records are not coordinate sorted")
    return keep.view(np.bool_)


def compact_reads(reads: ReadColumns, keep: np.ndarray) -> ReadColumns:
    """Admitted records only, repacked (host packer step; C++ because the payload columns are GB-sized)."""
    keep8 = np.ascontiguousarray(keep, dtype=np.uint8)
    n = int(keep8.sum())
    if n == reads.n:
        return reads
    if n == 0:
        return ReadColumns.empty()
    src = _lib.ReadBatch(reads.n, reads.n_cigar, reads.n_qual, _ptr(reads.pos), _ptr(reads.flag), _ptr(reads.mapq),
                         _ptr(reads.cigar_off), _ptr(reads.cigar), _ptr(reads.qual_off), _ptr(reads.qual))
    pos = np.empty(n, np.int32); flag = np.empty(n, np.uint16); mapq = np.empty(n, np.uint8)
    coff = np.empty(n + 1, np.uint32); cig = np.empty(max(reads.n_cigar, 1), np.uint32)
    qoff = np.empty(n + 1, np.uint64); qual = np.empty(max(reads.n_qual, 1), np.uint8)
    out = _lib.ReadBatch()
    rc = _lib.lib().clb_compact_reads(C.byref(src), _ptr(keep8), _ptr(pos), _ptr(flag), _ptr(mapq), _ptr(coff), _ptr(cig),
                                      _ptr(qoff), _ptr(qual), C.byref(out))
    if rc != 0:
        raise ClbError(rc, "clb_compact_reads failed")
    name_id = None if reads.name_id is None else reads.name_id[keep8.astype(bool)]
    return ReadColumns(pos, flag, mapq, coff, cig[: int(out.n_cigar)], qoff, qual[: int(out.n_qual)], name_id)


def count_unique_reads(reads: ReadColumns, keep: np.ndarray, length: int) -> int:
    """ContigProfiler.n_reads: distinct QNAMEs among admitted records that appear in >= 1 column
    (contig_profiler.rs:59-62).  Stays on the host (SURVEY.md H7)."""
    if reads.n == 0 or reads.name_id is None:
        return 0
    span = reads.ref_len()
    seen = keep & (span > 0) & (reads.pos.astype(np.int64) < length)
    return int(np.unique(reads.name_id[seen]).shape[0])


def bin_geometry(name: str, length: int, largest: int) -> Tuple[int, int]:
    s = C.c_uint32(0); n = C.c_uint32(0)
    _lib.lib().clb_bin_geometry(name.encode(), int(length), int(largest), C.byref(s), C.byref(n))
    return int(s.value), int(n.value)


def stitch_intervals(shards: Sequence[np.ndarray]) -> np.ndarray:
    """Concatenate region shards of one contig in genomic order, merging runs across soft seams."""
    shards = [np.ascontiguousarray(s, dtype=INTERVAL_DTYPE) for s in shards]
    total = sum(s.shape[0] for s in shards)
    out = np.zeros(total, dtype=INTERVAL_DTYPE)
    ptrs = (C.c_void_p * len(shards))(*[s.ctypes.data for s in shards])
    counts = (C.c_uint64 * len(shards))(*[s.shape[0] for s in shards])
    n = _lib.lib().clb_stitch_intervals(ptrs, counts, len(shards), _ptr(out))
    return out[: int(n)]


@dataclass
class ContigProfiler:
    """Per-contig sums; field names as in contig_profiler.rs:10-16."""
    name: str
    length: int
    n_covered_bases: int = 0
    summed_coverage: int = 0
    summed_baseq: int = 0
    summed_mapq: int = 0
    quality_bases: int = 0
    n_reads: int = 0
    bins: Optional[np.ndarray] = None
    stride: int = 0


class BedGraphWriter:
    """Depth runs (raw or QC) as bedGraph text (clb_bedgraph_writer): "name\tstart\tend\tdepth" lines, contigs in the order
    added."""

    def __init__(self, path: Optional[str]):
        self._L = _lib.lib()
        self.path = path
        self._w = self._L.clb_bedgraph_writer_open(path.encode() if path else None)
        if not self._w:
            raise ClbError(_lib.CLB_E_IO, f"cannot create {path}")

    def add_contig(self, name: str, length: int, runs: np.ndarray):
        r = np.ascontiguousarray(runs, dtype=RUN_DTYPE)
        rc = self._L.clb_bedgraph_writer_add_contig(self._w, name.encode(), int(length), _ptr(r), r.shape[0])
        if rc != 0:
            raise ClbError(rc, f"cannot write {self.path}" if rc == _lib.CLB_E_IO else f"depth runs of {name} do not tile [0,{length})")

    def text(self) -> bytes:
        n = C.c_uint64(0)
        p = self._L.clb_bedgraph_writer_buffer(self._w, C.byref(n))
        return C.string_at(p, n.value) if n.value else b""

    def close(self):
        if self._w:
            w, self._w = self._w, None
            rc = self._L.clb_bedgraph_writer_close(w)
            if rc != 0:
                raise ClbError(rc, f"cannot write {self.path}")

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class CallableProfiler:
    """BED writer + per-contig state counts that lives across contigs, like the reference's
    CallableProfiler (one instance per run; callable_profiler.rs:11-37)."""

    def __init__(self, bed_file: Optional[str], largest_contig_length: int):
        self._L = _lib.lib()
        self.bed_file = bed_file
        self.largest_contig_length = int(largest_contig_length)
        self._w = self._L.clb_bed_writer_open(bed_file.encode() if bed_file else None, self.largest_contig_length)
        if not self._w:
            raise ClbError(_lib.CLB_E_IO, f"cannot create {bed_file}")
        self.contig_counts: Dict[str, np.ndarray] = {}
        self._closed = False

    def add_contig(self, name: str, length: int, intervals: np.ndarray, state_counts, bins: Optional[np.ndarray], stride: int):
        iv = np.ascontiguousarray(intervals, dtype=INTERVAL_DTYPE)
        b = None if bins is None or bins.size == 0 else np.ascontiguousarray(bins, dtype=np.uint32)
        has = C.c_int(0)
        rc = self._L.clb_bed_writer_add_contig(self._w, name.encode(), int(length), _ptr(iv), iv.shape[0], _ptr(b),
                                               0 if b is None else b.shape[1], int(stride), C.byref(has))
        if rc != 0:
            raise ClbError(rc, f"cannot write {self.bed_file}" if rc == _lib.CLB_E_IO else f"intervals of {name} do not tile [0,{length})")
        self.contig_counts[name] = np.array(state_counts, dtype=np.uint64)
        return (b if has.value else None)

    def get_contig_counts(self, contig: str) -> np.ndarray:
        return self.contig_counts.get(contig, np.zeros(6, np.uint64))

    def bed_bytes(self) -> bytes:
        n = C.c_uint64(0)
        p = self._L.clb_bed_writer_buffer(self._w, C.byref(n))
        return C.string_at(p, n.value) if n.value else b""

    def close(self):
        if not self._closed:
            self._closed = True
            rc = self._L.clb_bed_writer_close(self._w)
            if rc != 0:
                raise ClbError(rc, f"cannot write {self.bed_file}")

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def process_single_contig(ctx: CallableLociContext, reads: ReadColumns, ref, counter: CallableProfiler,
                          contig_stats: Dict[int, ContigProfiler], options: CallableOptions, tid: int,
                          batch_reads: int = 0) -> ContigDeviceResult:
    """GPU drop-in for callable_loci::process_single_contig (mod.rs:44-147).

    ``reads`` are the contig's records in BAM order (what bam.fetch((tid,0,len)) yields); ``ref`` is the
    contig's reference (ASCII).  Admission and unique-name counting run on the host, everything per-base
    on the device; results are folded into ``counter`` and ``contig_stats[tid]`` like the reference does.
    """
    stats = contig_stats[tid]
    keep = admit_reads(reads, options.pileup_max_depth, tid)
    stats.n_reads = count_unique_reads(reads, keep, stats.length)
    admitted = compact_reads(reads, keep)
    ctx.begin_contig(tid, stats.name, stats.length, ref, counter.largest_contig_length, max_ref_span=admitted.max_ref_span())
    if batch_reads and admitted.n > batch_reads:
        ctx.reserve(admitted.n, admitted.n_cigar, admitted.n_qual)
        for lo in range(0, admitted.n, batch_reads):
            ctx.push_reads(admitted.slice(lo, lo + batch_reads))
    else:
        ctx.push_reads(admitted)
    res = ctx.finish_contig()
    stats.n_covered_bases = res.n_covered_bases
    stats.summed_coverage = res.summed_coverage
    stats.summed_baseq = res.summed_baseq
    stats.summed_mapq = res.summed_mapq
    stats.quality_bases = res.quality_bases
    stats.stride = res.stride
    stats.bins = counter.add_contig(stats.name, stats.length, res.intervals, res.state_counts, res.bins, res.stride)
    return res
