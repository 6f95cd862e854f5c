"""ctypes binding of the C-ABI library (include/callable_loci_b200.h).

The product path has NO CPU fallback: if the CUDA library is missing or no device is present the
calls below raise.  Only the host-half functions (admission, BED writer, stitching) work without a GPU.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CLB_LIB") or os.path.join(_HERE, "libcallable_loci_b200.so")

CLB_OK = 0
CLB_E_IO = -5
ERRORS = {-1: "CLB_E_INVALID", -2: "CLB_E_CUDA", -3: "CLB_E_INPUT", -4: "CLB_E_UNSUPPORTED", -5: "CLB_E_IO"}


class ClbError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"{ERRORS.get(code, code)}: {msg}")
        self.code = code


class Options(C.Structure):
    _fields_ = [("min_depth", C.c_uint32), ("max_depth", C.c_uint32), ("min_depth_for_low_mapq", C.c_uint32),
                ("min_mapping_quality", C.c_uint8), ("min_base_quality", C.c_uint8), ("max_low_mapq", C.c_uint8),
                ("_pad", C.c_uint8), ("max_low_mapq_fraction", C.c_double)]


class ReadBatch(C.Structure):
    _fields_ = [("n_reads", C.c_uint64), ("n_cigar", C.c_uint64), ("n_qual", C.c_uint64),
                ("pos", C.c_void_p), ("flag", C.c_void_p), ("mapq", C.c_void_p), ("cigar_off", C.c_void_p),
                ("cigar", C.c_void_p), ("qual_off", C.c_void_p), ("qual", C.c_void_p)]


class Interval(C.Structure):
    _fields_ = [("start", C.c_uint32), ("end", C.c_uint32), ("state", C.c_uint8), ("soft_start", C.c_uint8),
                ("_pad", C.c_uint16)]


class ContigResult(C.Structure):
    _fields_ = [("state_counts", C.c_uint64 * 6), ("n_covered_bases", C.c_uint64), ("summed_coverage", C.c_uint64),
                ("summed_baseq", C.c_uint64), ("summed_mapq", C.c_uint64), ("quality_bases", C.c_uint64),
                ("n_intervals", C.c_uint64), ("intervals", C.POINTER(Interval)), ("n_bins", C.c_uint32),
                ("stride", C.c_uint32), ("bins", C.POINTER(C.c_uint32)), ("region_start", C.c_uint32),
                ("region_end", C.c_uint32), ("kernel_ms", C.c_float), ("h2d_ms", C.c_float), ("pileup_ms", C.c_float), ("fast_ms", C.c_float),
                ("h2d_bytes", C.c_uint64),
                ("d2h_bytes", C.c_uint64), ("gpu_launches", C.c_uint32), ("general_windows", C.c_uint32),
                ("upload_ms", C.c_float), ("_pad", C.c_float)]


# every symbol include/callable_loci_b200.h declares (tests check that the library exports all of them)
SYMBOLS = [
    "clb_abi_version", "clb_device_count", "clb_window_positions", "clb_create", "clb_destroy", "clb_last_error", "clb_set_stream",
    "clb_begin_contig", "clb_reserve", "clb_push_reads", "clb_finish_contig", "clb_host_alloc", "clb_host_free", "clb_wait_uploads",
    "clb_rerun_resident",
    "clb_counters_device", "clb_refresh_counters", "clb_set_nccl_allreduce", "clb_allreduce_nccl", "clb_debug_per_base",
    "clb_set_depth_histogram", "clb_depth_histogram", "clb_set_depth_tiles", "clb_depth_tiles", "clb_set_depth_runs", "clb_depth_runs",
    "clb_set_qc_depth_runs", "clb_qc_depth_runs",
    "clb_set_depth_thresholds", "clb_depth_tile_thresholds",
    "clb_admit_reads", "clb_admit_reads_mt", "clb_admitter_new", "clb_admitter_push", "clb_admitter_free", "clb_compact_reads", "clb_bed_writer_open", "clb_bed_writer_add_contig", "clb_bed_writer_buffer",
    "clb_bed_writer_close", "clb_stitch_intervals", "clb_bin_geometry",
    "clb_bedgraph_writer_open", "clb_bedgraph_writer_add_contig", "clb_bedgraph_writer_buffer", "clb_bedgraph_writer_close",
]

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C decodingustools_b200/csrc`).  There is no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, u32, u64, i32 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int32
    L.clb_abi_version.restype = C.c_int
    L.clb_device_count.restype = C.c_int
    L.clb_window_positions.restype = C.c_uint32
    L.clb_create.restype = vp
    L.clb_create.argtypes = [C.c_int, C.POINTER(Options), C.c_char_p, C.c_size_t]
    L.clb_destroy.argtypes = [vp]
    L.clb_last_error.restype = C.c_char_p
    L.clb_last_error.argtypes = [vp]
    L.clb_set_stream.argtypes = [vp, vp]
    L.clb_begin_contig.argtypes = [vp, i32, C.c_char_p, u32, vp, u64, C.c_int, u32, u32, u32, u32]
    L.clb_reserve.argtypes = [vp, u64, u64, u64]
    L.clb_push_reads.argtypes = [vp, C.POINTER(ReadBatch)]
    L.clb_finish_contig.argtypes = [vp, C.POINTER(ContigResult)]
    L.clb_rerun_resident.argtypes = [vp, C.POINTER(ContigResult), C.POINTER(C.c_float)]
    L.clb_counters_device.argtypes = [vp, C.POINTER(vp), C.POINTER(u64)]
    L.clb_refresh_counters.argtypes = [vp, C.POINTER(ContigResult)]
    L.clb_allreduce_nccl.argtypes = [vp, vp]
    L.clb_set_nccl_allreduce.argtypes = [vp]
    L.clb_debug_per_base.argtypes = [vp, vp, vp, vp, vp]
    L.clb_set_depth_histogram.argtypes = [vp, u32]
    L.clb_depth_histogram.argtypes = [vp, C.POINTER(C.POINTER(u64)), C.POINTER(C.POINTER(u64)), C.POINTER(u32)]
    L.clb_set_depth_tiles.argtypes = [vp, u32]
    L.clb_depth_tiles.argtypes = [vp] + [C.POINTER(C.POINTER(u64))] * 4 + [C.POINTER(u32), C.POINTER(u32)]
    L.clb_set_depth_runs.argtypes = [vp, C.c_int]
    L.clb_set_depth_thresholds.argtypes = [vp, C.POINTER(u32), u32]
    L.clb_depth_tile_thresholds.argtypes = [vp, C.POINTER(C.POINTER(u64)), C.POINTER(C.POINTER(u64)), C.POINTER(C.POINTER(u32)),
                                            C.POINTER(u32), C.POINTER(u32)]
    L.clb_depth_runs.argtypes = [vp, C.POINTER(vp), C.POINTER(u64)]
    L.clb_set_qc_depth_runs.argtypes = [vp, C.c_int]
    L.clb_qc_depth_runs.argtypes = [vp, C.POINTER(vp), C.POINTER(u64)]
    L.clb_admit_reads.argtypes = [i32, u32, u64, vp, vp, vp, vp, vp]
    L.clb_host_alloc.restype = vp
    L.clb_host_alloc.argtypes = [C.c_size_t]
    L.clb_host_free.argtypes = [vp]
    L.clb_wait_uploads.argtypes = [vp]
    L.clb_admitter_new.restype = vp
    L.clb_admitter_new.argtypes = [i32, u32]
    L.clb_admitter_push.argtypes = [vp, i32, C.c_uint16, vp, u32]
    L.clb_admitter_free.argtypes = [vp]
    L.clb_admit_reads_mt.argtypes = [i32, u32, u64, vp, vp, vp, vp, u32, u32, vp, C.POINTER(u64)]
    L.clb_compact_reads.argtypes = [C.POINTER(ReadBatch), vp, vp, vp, vp, vp, vp, vp, vp, C.POINTER(ReadBatch)]
    L.clb_bed_writer_open.restype = vp
    L.clb_bed_writer_open.argtypes = [C.c_char_p, u32]
    L.clb_bed_writer_add_contig.argtypes = [vp, C.c_char_p, u32, vp, u64, vp, u32, u32, C.POINTER(C.c_int)]
    L.clb_bed_writer_buffer.restype = vp
    L.clb_bed_writer_buffer.argtypes = [vp, C.POINTER(u64)]
    L.clb_bed_writer_close.argtypes = [vp]
    L.clb_bedgraph_writer_open.restype = vp
    L.clb_bedgraph_writer_open.argtypes = [C.c_char_p]
    L.clb_bedgraph_writer_add_contig.argtypes = [vp, C.c_char_p, u32, vp, u64]
    L.clb_bedgraph_writer_buffer.restype = vp
    L.clb_bedgraph_writer_buffer.argtypes = [vp, C.POINTER(u64)]
    L.clb_bedgraph_writer_close.argtypes = [vp]
    L.clb_stitch_intervals.restype = u64
    L.clb_stitch_intervals.argtypes = [vp, vp, u32, vp]
    L.clb_bin_geometry.argtypes = [C.c_char_p, u32, u32, C.POINTER(u32), C.POINTER(u32)]
    _lib = L
    return L
