/*
 * callable_loci_b200.h -- C ABI of the B200-native CallableLoci hot path.
 *
 * This is the drop-in boundary for DecodingUsTools' `coverage` command.  The reference has no
 * FFI for this path: the seam is the Rust call
 *     callable_loci::process_single_contig(bam, fasta, header, counter, contig_stats, options, tid)
 *         (/root/reference/src/callable_loci/mod.rs:44-52, called from src/api/coverage.rs:238-252)
 * whose per-base pileup loop (mod.rs:65-142), classifier / run-length segmentation
 * (profilers/callable_profiler.rs:89-155), per-contig sums (profilers/contig_profiler.rs:47-83) and
 * bin counting (utils/histogram_plotter.rs:74-102) this library replaces.  A Rust host keeps BGZF/BAM
 * decode, htslib's read admission (A0), unique-QNAME counting and all text output, and binds the
 * functions below in an `extern "C"` block (see INTEGRATION.md).
 *
 * Conventions: plain pointers and sizes only; every function returns 0 on success or a negative
 * CLB_E_* code (message via clb_last_error); no exceptions cross the ABI; a context is bound to one
 * CUDA device and must be used from one thread at a time; result buffers are owned by the context
 * and stay valid until the next clb_begin_contig / clb_destroy on that context.
 */
#ifndef CALLABLE_LOCI_B200_H
#define CALLABLE_LOCI_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CLB_ABI_VERSION 2

enum {
    CLB_OK = 0,
    CLB_E_INVALID = -1,     /* bad argument / call order                               */
    CLB_E_CUDA = -2,        /* CUDA runtime error (no device, OOM, launch failure)     */
    CLB_E_INPUT = -3,       /* malformed columns: unsorted pos, offsets not monotone or not
                               starting at 0 (a read that runs past the contig / region end
                               is not an error: it is clipped there)                    */
    CLB_E_UNSUPPORTED = -4, /* a window's candidate reads span more than 4 GiB of qualities; NCCL not available */
    CLB_E_IO = -5
};

/* CalledState discriminants: /root/reference/src/callable_loci/types.rs:36-43 */
enum {
    CLB_REF_N = 0, CLB_CALLABLE = 1, CLB_NO_COVERAGE = 2, CLB_LOW_COVERAGE = 3,
    CLB_EXCESSIVE_COVERAGE = 4, CLB_POOR_MAPPING_QUALITY = 5
};

/* CallableOptions: /root/reference/src/callable_loci/options.rs:2-11 (selected_contigs stays on the host);
 * defaults /root/reference/src/cli.rs:34-60. */
typedef struct clb_options {
    uint32_t min_depth;               /* 4    */
    uint32_t max_depth;               /* 500  */
    uint32_t min_depth_for_low_mapq;  /* 10   */
    uint8_t  min_mapping_quality;     /* 10   */
    uint8_t  min_base_quality;        /* 20   */
    uint8_t  max_low_mapq;            /* 1    */
    uint8_t  _pad;
    double   max_low_mapq_fraction;   /* 0.1  */
} clb_options;

/* One column batch of decoded BAM records of the current contig: coordinate sorted, already
 * admission-filtered (clb_admit_reads), host memory (pinned memory makes the copies asynchronous).
 * Replaces what bam::IndexedReader::fetch + pileup() feed the reference (mod.rs:54-55). */
typedef struct clb_read_batch {
    uint64_t        n_reads;
    uint64_t        n_cigar;     /* == cigar_off[n_reads] - cigar_off[0] */
    uint64_t        n_qual;      /* == qual_off[n_reads]  - qual_off[0]  */
    const int32_t  *pos;         /* [n_reads]    0-based leftmost coordinate                      */
    const uint16_t *flag;        /* [n_reads]    BAM FLAG (0x4 records are skipped)               */
    const uint8_t  *mapq;        /* [n_reads]                                                     */
    const uint32_t *cigar_off;   /* [n_reads+1]  offsets into cigar[], relative to this batch     */
    const uint32_t *cigar;       /* [n_cigar]    BAM ops, len<<4|op                               */
    const uint64_t *qual_off;    /* [n_reads+1]  byte offsets into qual[], relative to this batch */
    const uint8_t  *qual;        /* [n_qual]     raw phred bytes                                  */
} clb_read_batch;

/* One BED run, half-open [start,end): callable_profiler.rs:42-46,131-150. */
typedef struct clb_interval {
    uint32_t start;
    uint32_t end;
    uint8_t  state;      /* CLB_* state                                                             */
    uint8_t  soft_start; /* 1: first run of a region shard whose state equals the base before the
                            shard (merge with the previous shard's last run when stitching)          */
    uint16_t _pad;
} clb_interval;

/* Everything process_single_contig accumulates for one contig (or one region shard of it):
 * state counts callable_profiler.rs:124-126; sums contig_profiler.rs:64-82; bins histogram_plotter.rs:74-102
 * (own positions only: the host adds quirk Q2's stale range, see clb_bed_writer_*). */
typedef struct clb_contig_result {
    uint64_t state_counts[6];
    uint64_t n_covered_bases;
    uint64_t summed_coverage;    /* == pileup cells == aligned bases processed */
    uint64_t summed_baseq;
    uint64_t summed_mapq;
    uint64_t quality_bases;
    uint64_t n_intervals;
    const clb_interval *intervals;   /* [n_intervals], ascending start, tiles [region_start, region_end) */
    uint32_t n_bins;                 /* contig_len / stride + 1 */
    uint32_t stride;
    const uint32_t *bins;            /* [3][n_bins]: CALLABLE, POOR_MAPPING_QUALITY, REF_N */
    uint32_t region_start;
    uint32_t region_end;
    float    kernel_ms;              /* device time of the pileup/classify/segment kernels (CUDA events) */
    float    h2d_ms;                 /* device time of the host->device copies                          */
    float    pileup_ms;              /* device time of the pileup kernels (k_pileup_fast + k_pileup_general) alone;
                                        only set by clb_rerun_resident                                  */
    float    fast_ms;                /* of which k_pileup_fast (the dominant kernel); clb_rerun_resident only */
    uint64_t h2d_bytes;
    uint64_t d2h_bytes;
    uint32_t gpu_launches;           /* kernels launched for this contig */
    uint32_t general_windows;        /* windows that took the general kernel (long CIGARs, deep piles, shard starts) */
    float    upload_ms;              /* device time of the upload-time helper kernels (offset validation / rebasing, read ends and
                                        CIGAR checkpoints of long reads, N-mask packing); part of kernel_ms, not of a resident re-run */
    float    _pad;
} clb_contig_result;

typedef struct clb_ctx clb_ctx;

/* ---------------------------------------------------------------- device path */
int         clb_abi_version(void);
int         clb_device_count(void);
/* Reference positions owned by one CTA window (region shards are best cut at multiples of it). */
uint32_t    clb_window_positions(void);
/* Create a context on `device`.  On failure returns NULL and writes a message to err (if non-NULL). */
clb_ctx    *clb_create(int device, const clb_options *opt, char *err, size_t err_len);
void        clb_destroy(clb_ctx *ctx);
const char *clb_last_error(const clb_ctx *ctx);
/* Run the kernels on a caller-owned cudaStream_t (NULL = the context's own stream). */
int         clb_set_stream(clb_ctx *ctx, void *cuda_stream);

/* Start a contig (or a region shard [region_start, region_end) of it; pass 0, contig_len for all).
 * ref: reference bases of the WHOLE contig; ref_kind 0 = ASCII bytes (ref_len bytes, bases past
 * ref_len read as 'N', mod.rs:79-80), 1 = bit-packed N-mask (uint32 words, bit p&31 of word p>>5,
 * ceil(contig_len/32)+1 words).  largest_contig_len: api/coverage.rs:210-215 (largest selected
 * non-chrM contig; drives the bin stride).  max_ref_span: upper bound of the reference span of any
 * read that will be pushed (0 = let the library compute it on the device). */
int clb_begin_contig(clb_ctx *ctx, int32_t tid, const char *name, uint32_t contig_len,
                     const void *ref, uint64_t ref_len, int ref_kind, uint32_t largest_contig_len,
                     uint32_t region_start, uint32_t region_end, uint32_t max_ref_span);
/* Optional capacity hint for the contig's totals (avoids device reallocation while streaming). */
int clb_reserve(clb_ctx *ctx, uint64_t n_reads, uint64_t n_cigar, uint64_t n_qual);
/* Append a batch (ascending pos across batches).  Copies are enqueued asynchronously; windows whose
 * reads have all arrived are launched right away so copy and compute overlap. */
int clb_push_reads(clb_ctx *ctx, const clb_read_batch *batch);
/* Finish the contig: remaining windows, interval compaction, device->host copy of the result. */
int clb_finish_contig(clb_ctx *ctx, clb_contig_result *out);
/* Page-locked host memory for column batches (copies from it are asynchronous and run at full PCIe speed), and a wait for
 * every copy queued so far, after which the pushed buffers may be reused. */
void *clb_host_alloc(size_t bytes);
void  clb_host_free(void *p);
int   clb_wait_uploads(clb_ctx *ctx);

/* Re-run all kernels of the current (finished) contig on the data already resident in HBM and
 * refresh the result; *ms receives the device time.  This is the HBM-resident measurement path.
 * With out == NULL and ms == NULL the kernels are only ENQUEUED on the context's compute stream (no host
 * synchronisation): steps, and a clb_allreduce_nccl after each, can be queued back to back and waited for once. */
int clb_rerun_resident(clb_ctx *ctx, clb_contig_result *out, float *ms);

/* Multi-GPU: the additive part of the result (11 counters + 3*n_bins bins, all uint64) lives in one
 * contiguous device buffer so the host can sum it across ranks (ncclAllReduce(ncclSum, ncclUint64) or
 * torch.distributed.all_reduce) and then re-read it with clb_refresh_counters. */
int clb_counters_device(clb_ctx *ctx, void **dev_ptr, uint64_t *n_u64);
int clb_refresh_counters(clb_ctx *ctx, clb_contig_result *out);
/* Same reduction done inside the library on an ncclComm_t the host created: one ncclAllReduce(ncclSum, ncclUint64) over
 * the counter buffer, enqueued on the context's compute stream (clb_refresh_counters synchronises).  The library does
 * not link NCCL: it calls the ncclAllReduce the host registered with clb_set_nccl_allreduce (the address of that
 * function in the NCCL build that created the communicator), else the first one visible in the process. */
int clb_set_nccl_allreduce(void *nccl_allreduce_fn);
int clb_allreduce_nccl(clb_ctx *ctx, void *nccl_comm);

/* Depth histograms (not in the reference; off by default).  n_bins = 0: off; else 2..65536.  Bin d counts the region's
 * positions that are not REF_N with depth d; the last bin counts depth >= n_bins - 1.  Takes effect at the next
 * clb_begin_contig; CLB_E_INVALID while a contig is open or when out of range.
 * Raw depth is the depth of summed_coverage (deletions and ref-skips included), QC depth the one of quality_bases (MAPQ >=
 * min_mapping_quality and base quality >= min_base_quality).  When on, both follow the bins in the counter buffer
 * ([12 counters][3 x n_bins bins][raw][qc], all counted by clb_counters_device), so region shards sum like the bins. */
int clb_set_depth_histogram(clb_ctx *ctx, uint32_t n_bins);
/* Raw-depth and QC-depth histograms of the last clb_finish_contig / clb_rerun_resident / clb_refresh_counters, [n_bins]
 * each, owned by the context like the other results.  When off: *n_bins = 0 and NULL pointers. */
int clb_depth_histogram(const clb_ctx *ctx, const uint64_t **raw, const uint64_t **qc, uint32_t *n_bins);

/* Depth tiles (not in the reference; off by default): a fixed grid of tile_len positions in whole-contig coordinates, tile t
 * = [t * tile_len, min((t + 1) * tile_len, contig_len)), n_tiles = ceil(contig_len / tile_len).  tile_len = 0: off; else
 * 256..2^31.  Per tile, over the region's positions in it: territory (positions that are not REF_N), callable (positions
 * classified CALLABLE), raw_sum and qc_sum (raw / QC depth summed over the positions that are not REF_N; depths as in the
 * depth histograms).  Mean depths are sum / territory.  Takes effect at the next clb_begin_contig; CLB_E_INVALID while a
 * contig is open or when out of range.  When on, the four arrays follow the histograms in the counter buffer
 * ([12 counters][3 x n_bins bins][hist raw][hist qc][territory][callable][raw_sum][qc_sum], all counted by
 * clb_counters_device), so region shards of one contig sum into the same tiles. */
int clb_set_depth_tiles(clb_ctx *ctx, uint32_t tile_len);
/* The tiles of the last clb_finish_contig / clb_rerun_resident / clb_refresh_counters, [n_tiles] each, owned by the context
 * like the other results.  When off: *n_tiles = 0, *tile_len = 0 and NULL pointers. */
int clb_depth_tiles(const clb_ctx *ctx, const uint64_t **territory, const uint64_t **callable, const uint64_t **raw_sum,
                    const uint64_t **qc_sum, uint32_t *n_tiles, uint32_t *tile_len);

/* Depth runs (not in the reference; off by default; like bedtools genomecov -bga or mosdepth's per-base output): the raw
 * depth of every position of [region_start, region_end) as runs of equal depth.  Raw depth is the depth of
 * summed_coverage: admitted reads whose reference span covers the position, deletions and ref-skips included, no MAPQ or
 * base-quality filter; REF_N positions and depth 0 are included.  Run i covers [start_i, start_{i+1}), the last one ends at
 * region_end; starts ascend strictly from region_start and adjacent runs differ in depth.
 * Region shards of one contig stitch by concatenation in genomic order, dropping a shard's first run when its depth equals
 * the previous shard's last (runs are defined by depth alone: no soft flag is needed). */
typedef struct clb_depth_run {
    uint32_t start;
    uint32_t depth;
} clb_depth_run;
/* on != 0: compute the runs from the next clb_begin_contig on; CLB_E_INVALID while a contig is open. */
int clb_set_depth_runs(clb_ctx *ctx, int on);
/* The runs of the last clb_finish_contig / clb_rerun_resident with a result, owned by the context like the intervals.
 * When off: *runs = NULL, *n_runs = 0.  d2h_bytes counts their copy. */
int clb_depth_runs(const clb_ctx *ctx, const clb_depth_run **runs, uint64_t *n_runs);

/* Debug/parity: copy the per-base counters of [region_start, region_end) (computed by a separate
 * un-fused launch of the same pileup code).  Each pointer may be NULL. */
int clb_debug_per_base(clb_ctx *ctx, uint32_t *raw, uint32_t *qc, uint32_t *low, uint8_t *state);

/* ---------------------------------------------------------------- host path (no GPU needed) */
/* htslib bam_plp_push admission as configured by the reference (mod.rs:55-60): keep[i] = 1 iff record i
 * enters the pileup.  maxcnt = max_depth > 0 ? max_depth : 500.  Returns CLB_E_INPUT if pos is unsorted. */
int clb_admit_reads(int32_t tid, uint32_t maxcnt, uint64_t n_reads, const int32_t *pos, const uint16_t *flag,
                    const uint32_t *cigar_off, const uint32_t *cigar, uint8_t *keep);

/* Same result on n_threads host threads (0 = all cores, at most 16).  Only records that have at least maxcnt records
 * starting within max_ref_span before them can be refused; the others are decided independently, the rest is replayed
 * sequentially run by run.  max_ref_span: upper bound of any record's reference span (0 = compute it here).
 * *n_replayed (may be NULL) receives how many records went through the sequential recurrence (0 on ordinary 30x data). */
int clb_admit_reads_mt(int32_t tid, uint32_t maxcnt, uint64_t n_reads, const int32_t *pos, const uint16_t *flag,
                       const uint32_t *cigar_off, const uint32_t *cigar, uint32_t max_ref_span, uint32_t n_threads,
                       uint8_t *keep, uint64_t *n_replayed);

/* The same decision one record at a time, for a decoder that packs only admitted records: returns 1 (admitted), 0
 * (refused or unmapped) or a negative CLB_E_* code (records out of order).  One admitter per contig. */
typedef struct clb_admitter clb_admitter;
clb_admitter *clb_admitter_new(int32_t tid, uint32_t maxcnt);
int           clb_admitter_push(clb_admitter *a, int32_t pos, uint16_t flag, const uint32_t *cigar, uint32_t n_cigar);
void          clb_admitter_free(clb_admitter *a);

/* Drop the records with keep[i] == 0 and repack the columns (what the host packer does after admission).
 * Output buffers must be at least as large as the inputs; offsets are rebased to start at 0.
 * out->n_reads / n_cigar / n_qual receive the compacted sizes. */
int clb_compact_reads(const clb_read_batch *in, const uint8_t *keep, int32_t *pos, uint16_t *flag, uint8_t *mapq,
                      uint32_t *cigar_off, uint32_t *cigar, uint64_t *qual_off, uint8_t *qual, clb_read_batch *out);

/* BED writer with the reference's cross-contig behaviour (quirks Q1/Q2): callable_profiler.rs:39-87,122-155. */
typedef struct clb_bed_writer clb_bed_writer;
clb_bed_writer *clb_bed_writer_open(const char *path /* NULL = in-memory */, uint32_t largest_contig_len);
/* Append one contig (ascending tid).  Intervals must tile [0, contig_len) (stitched shards).
 * bins_inout: [3][n_bins] from the device, updated in place with the stale range of the previous
 * contig (Q2); may be NULL.  *has_bins (may be NULL) receives whether the reference would have
 * produced a histogram for this contig (finish_contig, callable_profiler.rs:67). */
int  clb_bed_writer_add_contig(clb_bed_writer *w, const char *name, uint32_t contig_len,
                               const clb_interval *iv, uint64_t n_iv,
                               uint32_t *bins_inout, uint32_t n_bins, uint32_t stride, int *has_bins);
const char *clb_bed_writer_buffer(clb_bed_writer *w, uint64_t *len);   /* in-memory mode */
int  clb_bed_writer_close(clb_bed_writer *w);
/* bedGraph writer for depth runs: lines "name\tstart\tend\tdepth\n", no header.  Runs must tile [0, contig_len) (stitched
 * shards; none for an empty contig), else CLB_E_INVALID; a failed write gives CLB_E_IO.  A non-seekable path (a FIFO,
 * /dev/stdout) is written in order. */
typedef struct clb_bedgraph_writer clb_bedgraph_writer;
clb_bedgraph_writer *clb_bedgraph_writer_open(const char *path /* NULL = in-memory */);
int  clb_bedgraph_writer_add_contig(clb_bedgraph_writer *w, const char *name, uint32_t contig_len, const clb_depth_run *runs, uint64_t n);
const char *clb_bedgraph_writer_buffer(clb_bedgraph_writer *w, uint64_t *len);   /* in-memory mode */
int  clb_bedgraph_writer_close(clb_bedgraph_writer *w);
/* Concatenate region shards of one contig in genomic order, merging soft starts.  Returns the number
 * of intervals written to out (capacity must be >= sum of inputs). */
uint64_t clb_stitch_intervals(const clb_interval *const *shards, const uint64_t *n_per_shard, uint32_t n_shards,
                              clb_interval *out);
/* Bin stride and count: histogram_plotter.rs:424-431,75. */
int clb_bin_geometry(const char *name, uint32_t contig_len, uint32_t largest_contig_len,
                     uint32_t *stride, uint32_t *n_bins);

#ifdef __cplusplus
}
#endif
#endif /* CALLABLE_LOCI_B200_H */
