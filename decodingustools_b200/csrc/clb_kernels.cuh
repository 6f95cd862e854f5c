// clb_kernels.cuh -- hand-written sm_100a kernels of the CallableLoci hot path.
//
// Replaces the reference's per-base CPU loop:
//   htslib bam_plp64_next + process_position          /root/reference/src/callable_loci/mod.rs:17-42,65-120
//   CallableProfiler::process_position/process_state  .../profilers/callable_profiler.rs:89-155
//   ContigProfiler::process_position                  .../profilers/contig_profiler.rs:47-83
//   HistogramPlotter::process_coverage_ranges         .../utils/histogram_plotter.rs:74-102
//
// Design (see DESIGN.md): one CTA owns a reference window of WREAL positions plus one halo position
// to its left.  Warps take 32 candidate reads at a time (coalesced column loads), walk the CIGARs
// (lane-serial for short CIGARs, warp-cooperative prefix sums for long ones), and turn every read /
// M-segment into two shared-memory difference-array updates instead of one update per base.  The
// M-segments go to a CTA-wide pool; after a barrier all threads stream their base qualities once with
// 16-byte loads (prefetched into L2 at window start) and add one fail flag per byte to packed
// per-position counters.  After a block scan the window is classified, run boundaries are compacted
// into interval records, and counters / bins are reduced per CTA before a handful of global atomics.
// No per-base array ever reaches HBM.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <type_traits>

namespace clb {

#ifndef CLB_NT
#define CLB_NT 256
#endif
constexpr int NT = CLB_NT;            // threads per CTA
constexpr int NWARPS = NT / 32;
static_assert(NWARPS <= 32, "cross-warp prefixes are taken with one warp-wide reduction");
#ifndef CLB_PPT
#define CLB_PPT 8
#endif
#ifndef CLB_MINB
#define CLB_MINB 5
#endif
constexpr int PPT = CLB_PPT;          // window entries per thread in the classify phase
constexpr int WN = NT * PPT;          // entries per window; entry 0 is the halo position (window start - 1)
constexpr int WREAL = WN - 1;         // reference positions owned by one window
constexpr int MAXSEG = 2;             // M-like segments a "simple" read may contribute
constexpr int FAST_OPS = 6;           // CIGAR ops walked lane-serially; longer CIGARs go warp-cooperative
constexpr int NFIRST = 128;           // low-MAPQ threshold table entries cached in shared memory
#ifndef CLB_KLQ
#define CLB_KLQ 4
#endif
constexpr int KLQ = CLB_KLQ;          // packed-u8 low-BQ arrays per window
constexpr int BPA = 7;                // 32-read batches per packed array: 7 * 32 = 224 increments max < 256
constexpr int LQ_SLAB = WN / 4 + 32;   // words per packed array: 16 words of padding on both sides for clamped / straddling chunks
constexpr int NRCP = 160;             // reciprocal table size (slots per segment)
constexpr unsigned FULL = 0xffffffffu;
constexpr int STAT_STRIDE = 16;       // one 128-byte line per global counter (u64 units)

enum { ST_REF_N = 0, ST_CALLABLE = 1, ST_NO_COVERAGE = 2, ST_LOW_COVERAGE = 3, ST_EXCESSIVE = 4, ST_POOR_MAPQ = 5 };
enum { S_COUNT0 = 0, S_COVERED = 6, S_SUMCOV = 7, S_SUMBQ = 8, S_SUMMAPQ = 9, S_QBASES = 10, S_RESERVED = 11, N_STATS = 12 };
enum { ERR_QUAL_SPAN = 1, ERR_REC_OVERFLOW = 2, ERR_UNSORTED = 8, ERR_OFFSETS = 16 };
// k_validate_batch refused the columns: the pileup kernels do not walk them and return before writing win_tab[w]
constexpr uint32_t ERR_INPUT_REFUSED = ERR_UNSORTED | ERR_OFFSETS;
// the kernels after the pileup do not touch win_tab / rec once one of these is set: the input was refused or a window could
// not be run; the host reports the error instead
constexpr uint32_t ERR_RESULT_INVALID = ERR_INPUT_REFUSED | ERR_QUAL_SPAN;

constexpr int TH_MAX = 8;             // depth thresholds per tile grid (KParams::thr)

struct KParams {
    // packed read columns (device)
    const int32_t  *pos;
    const uint16_t *flag;
    const uint8_t  *mapq;
    const uint32_t *cigar_off;
    const uint32_t *cigar;
    const uint64_t *qual_off;
    const uint8_t  *qual;
    uint64_t qual_bytes;           // allocated extent of qual (bounds-checked builds)
    const uint32_t *read_end;      // optional (long-read mode): pos + reference span, else nullptr
    const uint2    *cigar_ckpt;    // optional (long-read mode): (reference, query) offset of the owning read at every 32nd CIGAR op
    // contig / region
    const uint32_t *nmask;         // bit-packed REF_N mask, zero padded past the contig end
    uint32_t region_start, region_end;
    // options
    uint32_t min_depth, max_depth, min_depth_for_low_mapq;
    uint32_t min_mapq, min_bq, max_low_mapq;
    const uint32_t *first_tab;     // [65536] smallest low count with low/raw > fraction (f64, exact)
    const uint8_t *first_tab8;     // [256] the same for raw depths below 256, one byte each (k_pileup_fast)
    const uint32_t *win_tables;    // WIN_TABLE_BYTES: the per-window shared-memory tables, ready to copy (k_window_tables)
    double max_low_mapq_fraction;  // for depths past the table (deep windows)
    // windows
    // per window, three 16-byte words (k_window_ranges): [0] candidate reads [x, y), first histogram bin z, window entry w where the
    // next bin starts; [1] quality bytes [lo (16-byte aligned), hi) of the candidate reads as two u64; [2] x = reads per warp
    // sub-batch of k_pileup_fast (0: general-path window), y = sub-batches, [z, w) = CIGAR ops of the candidate reads
    const uint4 *win_rec;
    uint32_t win_first;
    // outputs
    unsigned long long *stats;     // [N_STATS * STAT_STRIDE]
    unsigned long long *bins;      // [3][n_bins]
    uint32_t n_bins, stride;
    unsigned long long *rec;       // boundary records (pack_rec)
    uint32_t rec_cap;
    uint32_t *rec_cursor;
    uint2 *win_tab;                // per window: (first record, pack_win_y word)
    uint32_t *err;
    uint32_t *deep_count, *deep_list;   // windows with more than 65535 candidate reads, left to k_pileup_classify_deep
    uint32_t *gen_list, *gen_count, *gen_taken;   // queue of general-path windows (k_pileup_general takes tickets)
    const uint32_t *max_span;           // upper bound of the reference span of any read of the contig
    // optional per-base debug output, indexed by position - region_start
    uint32_t *dbg_raw, *dbg_qc, *dbg_low;
    uint8_t *dbg_state;
    long long *timing;             // optional (developer builds): 8 clock64 stamps per window
    // depth histograms (HIST instantiations only): DH_SLOTS copies of [raw n][qc n], CTA b adds to copy b % DH_SLOTS;
    // k_fold_depth_hist sums them into the counter buffer
    unsigned long long *dhist;
    uint32_t dh_n;                 // bins per histogram, 2 .. 65536; the last one counts every depth >= dh_n - 1
    // depth tiles (TILES instantiations only): [territory][callable][raw_sum][qc_sum], n_tiles u64 each, in the counter buffer.
    // Tile t covers contig positions [t * tile_len, min((t + 1) * tile_len, contig length)); tile_len >= 256.
    unsigned long long *tiles;
    uint32_t tile_len, n_tiles;
    // depth runs (RUNS instantiations): (position, raw depth) of every run start, reserved per window from run_cursor;
    // run_win_tab[w] = (first record, count | window soft << 16, raw depth of the first own entry, of the last one).  At most
    // one record per position: run_cap = region length.
    uint2 *run_rec;
    uint32_t *run_cursor;
    uint4 *run_win_tab;
    uint32_t run_cap;
    // depth thresholds (THRESH instantiations, always with TILES): thr[0 .. n_thr) strictly ascending, thr[n_thr ..] unused;
    // per tile the own positions that are not REF_N with raw / QC depth >= thr[j], at tiles + (4 + j) * n_tiles (raw) and
    // tiles + (4 + n_thr + j) * n_tiles (QC)
    uint32_t thr[TH_MAX];
    uint32_t n_thr;
    // QC depth runs (QRUNS instantiations): the depth runs keyed on the QC depth (the depth behind quality_bases) instead of
    // the raw depth.  (position, QC depth) records reserved per window from qrun_cursor; qrun_win_tab in run_win_tab's
    // format, with QC depths.  At most one record per position: qrun_cap = region length.
    uint2 *qrun_rec;
    uint32_t *qrun_cursor;
    uint4 *qrun_win_tab;
    uint32_t qrun_cap;
};

// The optional outputs of the pileup kernels (template argument FEAT); the instantiations with a feature are only launched
// when it is on, so the ones without stay as they were.  FEAT_THRESH is only instantiated together with FEAT_TILES.
enum : unsigned { FEAT_HIST = 1u, FEAT_TILES = 2u, FEAT_RUNS = 4u, FEAT_THRESH = 8u, FEAT_QRUNS = 16u };

// Developer builds only (scripts/phase_timing.py): slot i of window w's 8 timing words, written by thread 0 of a pileup
// kernel with P and w in scope.  The stamps cost instruction-cache space, so production builds compile them out.
#ifdef CLB_PHASE_TIMING
#define CLB_STAMP_VALUE(i, v) do { if (P.timing && threadIdx.x == 0) P.timing[(size_t)w * 8 + (i)] = (long long)(v); } while (0)
#else
#define CLB_STAMP_VALUE(i, v) do { } while (0)
#endif
#define CLB_STAMP(i) CLB_STAMP_VALUE(i, clock64())

// One bulk L2 prefetch of bytes [lo, hi) of a device array (rounded out to 16 bytes: allocations are 256-byte granular).
__device__ __forceinline__ void l2_prefetch(const void *base, uint64_t lo, uint64_t hi, uint32_t max_bytes) {
    const uint64_t a = ((uint64_t)(uintptr_t)base + lo) & ~15ull, b = ((uint64_t)(uintptr_t)base + hi + 15ull) & ~15ull;
    if (b <= a) return;
    const uint32_t bytes = (uint32_t)min(b - a, (uint64_t)max_bytes);
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" :: "l"(a), "r"(bytes) : "memory");
}

__device__ __forceinline__ uint4 ldg_stream(const uint4 *p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

__device__ __forceinline__ bool op_is_m(uint32_t op) { return op == 0 || op == 7 || op == 8; }
__device__ __forceinline__ bool op_ref(uint32_t op) { return op == 0 || op == 2 || op == 3 || op == 7 || op == 8; }
__device__ __forceinline__ bool op_qry(uint32_t op) { return op == 0 || op == 1 || op == 4 || op == 7 || op == 8; }

struct Seg { uint32_t qrel, rrel, len; };
// 8-byte segment descriptor: x = qrel; y = rrel (11 bits) | len (11) | chunks (8) | low-BQ slab (2)
static_assert(WN <= 2048 && KLQ <= 4, "descriptor bit fields");
__device__ __forceinline__ uint2 pack_desc(const Seg &s, uint32_t nc, uint32_t slab) {
    return make_uint2(s.qrel, s.rrel | (s.len << 11) | (nc << 22) | (slab << 30));
}

// Per-CTA constants; shared-memory arrays are addressed through 32-bit shared-window addresses
struct Win {
    long long wb, wend;            // position of entry 0, exclusive end of positions handled
    uint32_t n_ent;                // entries in use = wend - wb
    uint64_t qbase;                // 16-byte aligned byte offset of the window's first candidate quality
    const uint8_t *qual;
    uint64_t qual_bytes;
    uint32_t sA, sB;               // shared addresses of the difference arrays
    uint32_t sL;                   // deep windows only: low-MAPQ difference array (otherwise packed into the high half of sA)
    uint32_t min_bq, min_mapq, max_low_mapq;
    bool lq_packed;                // low-BQ counters: KLQ packed-u8 arrays (fast) or one u32 per position
};

__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// -DCLB_BOUNDS_CHECK (developer / test builds: compute-sanitizer is not available on the GPU pool this was developed on):
// every shared-memory atomic / vector load issued through the helpers below and every streamed quality load is checked
// against the extent it may touch; violations are counted in g_clb_bounds_violations (read with clb_debug_bounds) and the
// access is skipped.  Production builds compile the checks out.
__device__ unsigned int g_clb_bounds_violations;
#ifdef CLB_BOUNDS_CHECK
extern __shared__ __align__(16) uint8_t clb_smem_probe[];
__device__ __forceinline__ bool smem_ok(uint32_t saddr, uint32_t bytes) {
    uint32_t dyn; asm("mov.u32 %0, %%dynamic_smem_size;" : "=r"(dyn));
    const uint32_t base = smem_addr(clb_smem_probe);
    const bool ok = saddr >= base && saddr + bytes <= base + dyn && (saddr & (bytes - 1u)) == 0u;
    if (!ok) atomicAdd(&g_clb_bounds_violations, 1u);
    return ok;
}
#define CLB_SMEM_OK(a, n) smem_ok((a), (n))
#define CLB_GMEM_OK(p, lo, hi) (((const uint8_t *)(p) >= (const uint8_t *)(lo) && (const uint8_t *)(p) + 16 <= (const uint8_t *)(hi)) ? true : (atomicAdd(&g_clb_bounds_violations, 1u), false))
#else
#define CLB_SMEM_OK(a, n) true
#define CLB_GMEM_OK(p, lo, hi) true
#endif

__device__ __forceinline__ void red_shared(uint32_t saddr, uint32_t val) {
    if (!CLB_SMEM_OK(saddr, 4u)) return;
    asm volatile("red.shared.add.u32 [%0], %1;" :: "r"(saddr), "r"(val) : "memory");
}
// single-lane shared atomics as plain instructions (the compiler wraps atomicAdd/atomicMax in warp-aggregation code
// that is pure overhead when the caller has already elected one lane)
__device__ __forceinline__ uint32_t atom_shared_add(uint32_t saddr, uint32_t val) {
    uint32_t old = 0;
    if (!CLB_SMEM_OK(saddr, 4u)) return old;
    asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(saddr), "r"(val) : "memory");
    return old;
}
__device__ __forceinline__ void red_shared_max(uint32_t saddr, uint32_t val) {
    if (!CLB_SMEM_OK(saddr, 4u)) return;
    asm volatile("red.shared.max.u32 [%0], %1;" :: "r"(saddr), "r"(val) : "memory");
}
// add only when val != 0: one ISETP + one predicated ATOMS, no branch
__device__ __forceinline__ void red_shared_nz(uint32_t saddr, uint32_t val) {
    if (!CLB_SMEM_OK(saddr, 4u)) return;
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %1, 0;\n\t@p red.shared.add.u32 [%0], %1;\n\t}" :: "r"(saddr), "r"(val) : "memory");
}

// SWAR: 0x80 in every byte of x that is < T (unsigned).  t_low = (T & 0x7f) * 0x01010101; BQ_HI = (T >= 128).
template <bool BQ_HI>
__device__ __forceinline__ uint32_t bytes_lt(uint32_t x, uint32_t t_low) {
    const uint32_t H = 0x80808080u;
    const uint32_t d = (x | H) - t_low;                  // bit7 = ((x & 0x7f) >= (T & 0x7f)), no cross-byte borrow
    return BQ_HI ? (~(x & d) & H) : (~(x | d) & H);
}

// Difference-array update for one M-like segment (reads with mapq >= min_mapq only); returns the part of
// the segment inside the window proper (entries >= 1) as a Seg.  rel/qp: window entry (may be negative) and query
// offset of the op start; q0: absolute byte offset of the read's qualities; lq: its quality length.
__device__ __forceinline__ bool emit_m(const Win &W, uint32_t lq_arr, int rel, uint32_t qp, uint32_t len, uint64_t q0, uint32_t lq, Seg &out) {
    if (qp >= lq || rel >= (int)W.n_ent) return false;   // record.qual().get(qpos) == None / right of the window
    len = min(len, lq - qp);
    const uint32_t room = (uint32_t)((int)W.n_ent - rel);                       // > 0
    const uint32_t e1 = len >= room ? W.n_ent : (uint32_t)(rel + (int)len);     // exclusive end entry, clipped (rel + len may be <= 0)
    if ((int)e1 <= max(rel, 0)) return false;
    uint32_t e0 = (uint32_t)max(rel, 0);
    red_shared(W.sB + 4u * e0, 1u);
    red_shared_nz(W.sB + 4u * min(e1, (uint32_t)WN - 1u), e1 < (uint32_t)WN ? 0xffffffffu : 0u);
    if (e0 == 0) {                                       // covers the halo position: test its one base here
        const uint8_t q = W.qual[q0 + qp + (uint32_t)(-rel)];
        red_shared_nz(lq_arr + 64u, q < W.min_bq ? 1u : 0u);   // entry 0 = byte 0 of word 0 in both counter layouts
        e0 = 1;
        if (e1 <= 1) return false;
    }
    out.rrel = e0;
    out.len = e1 - e0;
    out.qrel = (uint32_t)(q0 - W.qbase) + qp + (uint32_t)((int)e0 - rel);
    return true;
}

// Difference-array update for a whole read (raw depth + low-MAPQ depth packed as lo16|hi16).  rel/rel_end: entries.
template <bool WIDE>
__device__ __forceinline__ void emit_read(const Win &W, int rel, int rel_end, uint32_t mq, unsigned long long &acc_mapq) {
    const int s = max(rel, 0), e = min(rel_end, (int)W.n_ent);
    if (e <= s) return;
    const uint32_t e0 = (uint32_t)s, e1 = (uint32_t)e;
    const bool lowq = mq <= W.max_low_mapq;
    const uint32_t delta = 1u + ((lowq && !WIDE) ? 0x10000u : 0u);
    const uint32_t o1 = 4u * min(e1, (uint32_t)WN - 1u);
    red_shared(W.sA + 4u * e0, delta);
    red_shared_nz(W.sA + o1, e1 < (uint32_t)WN ? 0u - delta : 0u);
    if (WIDE && lowq) {
        red_shared(W.sL + 4u * e0, 1u);
        red_shared_nz(W.sL + o1, e1 < (uint32_t)WN ? 0xffffffffu : 0u);
    }
    const uint32_t rs = max(e0, 1u);
    if (mq >= W.min_mapq && e1 > rs) acc_mapq += (unsigned long long)mq * (e1 - rs);
}

// One 16-byte quality chunk.  e0 = window entry of chunk byte 0 (may be < 0 or past the window for bytes outside
// [lo, hi), which are forced to 0xFF so they never fail and are subtracted from the sums).  Straight-line code:
// shared-memory atomics are cheaper on sm_100a (about one warp-wide ATOMS per clock per SM) than branches around them.
// LAYOUT: 1 = packed u8 low-BQ counters, 0 = one u32 per position, 2 = decided per window at run time (W.lq_packed)
template <bool BQ_HI, int LAYOUT>
__device__ __forceinline__ void process_chunk(const Win &W, uint32_t lq_arr, int e0, uint32_t lo, uint32_t hi, uint4 v, const uint4 *sMaskLo,
                                              const uint4 *sMaskHi, uint32_t t_low, uint32_t &acc_sum) {
    const uint4 ml = sMaskLo[lo], mh = sMaskHi[hi];       // 0xFF in bytes outside [lo, hi)
    v.x |= ml.x | mh.x; v.y |= ml.y | mh.y; v.z |= ml.z | mh.z; v.w |= ml.w | mh.w;
    const uint32_t l0 = bytes_lt<BQ_HI>(v.x, t_low), l1 = bytes_lt<BQ_HI>(v.y, t_low);        // 0x80 in every failing byte
    const uint32_t l2 = bytes_lt<BQ_HI>(v.z, t_low), l3 = bytes_lt<BQ_HI>(v.w, t_low);
    const uint32_t ONES = 0x01010101u;
    // dot products against the 0x80 flags give 128 x (count, sum) of the failing bytes
    const uint32_t tot = __dp4a(v.x, ONES, __dp4a(v.y, ONES, __dp4a(v.z, ONES, __dp4a(v.w, ONES, 0u))));
    const uint32_t sf128 = __dp4a(v.x, l0, __dp4a(v.y, l1, __dp4a(v.z, l2, __dp4a(v.w, l3, 0u))));
    const uint32_t ninv = lo + (16u - hi);
    acc_sum += tot - 255u * ninv - (sf128 >> 7);
    const uint32_t f0 = l0 >> 7, f1 = l1 >> 7, f2 = l2 >> 7, f3 = l3 >> 7;                    // 1 in every failing byte
    if (LAYOUT == 2 ? W.lq_packed : LAYOUT == 1) {
        // four positions per 32-bit word, one byte each: shift the 16 fail flags to the entry alignment and add them
        // with five unconditional atomics (a byte takes <= 224 increments, see BPA).
        const uint32_t sh = ((uint32_t)e0 & 3u) << 3;
        const uint32_t base = lq_arr + 64u + (uint32_t)((e0 >> 2) * 4);      // arrays start 16 words into their slab (e0 >= -15)
        red_shared(base + 0, f0 << sh);
        red_shared(base + 4, __funnelshift_l(f0, f1, sh));
        red_shared(base + 8, __funnelshift_l(f1, f2, sh));
        red_shared(base + 12, __funnelshift_l(f2, f3, sh));
        red_shared(base + 16, __funnelshift_l(f3, 0u, sh));
    } else {
        uint32_t m = f0 | (f1 << 1) | (f2 << 2) | (f3 << 3);      // bit (8*j + w) <=> chunk byte 4*w + j
        while (m) {
            const uint32_t b = __ffs(m) - 1; m &= m - 1;
            red_shared(lq_arr + 64u + 4u * (uint32_t)(e0 + (int)(((b & 7u) << 2) + (b >> 3))), 1u);
        }
    }
}

// Stream the qualities of the n_owner segments whose descriptors sit in desc[0..n_owner):
//   desc = pack_desc(segment, n_chunks, low-BQ slab).
// Every segment gets S2 slots of two consecutive chunks (S2 = ceil(largest chunk count / 2)), so slot f belongs to
// segment f / S2: no lookup table and no prefix sum; slots past a segment's end run empty.  The caller's threads
// cover slots f0, f0 + stride, ... (a warp: f0 = lane, stride 32; the whole CTA: f0 = tid, stride NT).
template <bool BQ_HI, int LAYOUT>
__device__ __forceinline__ void process_slots(const Win &W, uint32_t sLQ_s, uint32_t n_owner, uint32_t S2, const uint2 *desc,
                                              const uint32_t *sRcp, const uint4 *sMaskLo, const uint4 *sMaskHi, uint32_t t_low,
                                              uint32_t &acc_sum, uint32_t f0, uint32_t stride) {
    const uint8_t *P_qual_lo = W.qual, *P_qual_hi = W.qual + W.qual_bytes; (void)P_qual_lo; (void)P_qual_hi;
    const uint32_t total = n_owner * S2;
    const uint32_t rcp = S2 < (uint32_t)NRCP ? sRcp[S2] : 0xffffffffu / S2 + 1u;     // ceil(2^32 / S2): exact quotient for f < 2^32 / S2
    const uint8_t *qb = W.qual + W.qbase;
    for (uint32_t f = f0; f < total; f += stride) {
        const uint32_t o = S2 > 1 ? __umulhi(f, rcp) : f;
        const uint32_t c = 2u * (f - o * S2);
        const uint2 d = desc[o];
        const uint32_t head = d.x & 15u;
        const int rem = (int)(head + ((d.y >> 11) & 0x7ffu)) - (int)(16u * c);   // bytes from chunk c's start to the segment end
        if (rem <= 0) continue;
        const uint4 *src = reinterpret_cast<const uint4 *>(qb + (d.x & ~15u)) + c;
#ifdef CLB_EXPERIMENT_NOLOAD
        const uint4 v0 = make_uint4(0x25252525u + (uint32_t)(size_t)src, 0x25250225u, 0x25252525u, 0x25252525u), v1 = v0;   // timing experiment only
#else
        if (!CLB_GMEM_OK(src, P_qual_lo, P_qual_hi) || !CLB_GMEM_OK(src + 1, P_qual_lo, P_qual_hi)) continue;
        const uint4 v0 = ldg_stream(src);
        const uint4 v1 = ldg_stream(src + 1);                             // may lie past the segment (buffers are padded): masked below
#endif
        const int e0 = (int)((d.y & 0x7ffu) + 16u * c) - (int)head;
        const uint32_t lq_arr = sLQ_s + (d.y >> 30) * (uint32_t)(LQ_SLAB * 4);
        process_chunk<BQ_HI, LAYOUT>(W, lq_arr, e0, c == 0 ? head : 0u, (uint32_t)min(rem, 16), v0, sMaskLo, sMaskHi, t_low, acc_sum);
        if (rem > 16) process_chunk<BQ_HI, LAYOUT>(W, lq_arr, e0 + 16, 0u, (uint32_t)min(rem - 16, 16), v1, sMaskLo, sMaskHi, t_low, acc_sum);
    }
}

__device__ __forceinline__ uint32_t seg_chunks(const Seg &s) { return ((s.qrel & 15u) + s.len + 15u) >> 4; }

// Warp-collective: lanes holding a segment (has) publish it compactly into the warp's descriptor area and stream it
// right away (segments too long for the CTA pool, and the long-CIGAR path).
template <bool BQ_HI>
__device__ __forceinline__ void run_segments(const Win &W, uint32_t sLQ_s, uint32_t slab, bool has, const Seg &sg, uint2 *myDesc,
                                             const uint32_t *sRcp, const uint4 *sMaskLo, const uint4 *sMaskHi, uint32_t t_low,
                                             uint32_t &acc_sum, int lane) {
    const uint32_t bal = __ballot_sync(FULL, has);
    if (bal == 0) return;
    const uint32_t nc = has ? seg_chunks(sg) : 0u;
    const uint32_t S2 = (__reduce_max_sync(FULL, nc) + 1u) >> 1;
    if (has) myDesc[__popc(bal & ((1u << lane) - 1u))] = pack_desc(sg, nc, slab);
    __syncwarp();
    process_slots<BQ_HI, 2>(W, sLQ_s, __popc(bal), S2, myDesc, sRcp, sMaskLo, sMaskHi, t_low, acc_sum, (uint32_t)lane, 32u);
    __syncwarp();
}

// Warp-collective expansion of one long CIGAR: 32 ops per step (blocks aligned to 32 ops of the contig-wide CIGAR column),
// shuffle prefix sums over the (reference, query) lengths, one M-segment per lane streamed right away.  With checkpoints
// (k_cigar_checkpoints) the walk starts at the last block that begins at or left of the window instead of at the read start.
template <bool BQ_HI, bool WIDE>
__device__ __forceinline__ void expand_long_read(const Win &W, const KParams &P, uint32_t sLQ_s, uint32_t slab, int crel, uint32_t cmq,
                                                 uint32_t c0, uint32_t cn, uint32_t clq, uint64_t cq0, uint2 *myDesc, const uint32_t *sRcp,
                                                 const uint4 *sMaskLo, const uint4 *sMaskHi, uint32_t t_low, uint32_t &acc_sum,
                                                 unsigned long long &acc_mapq, int lane) {
    const uint32_t lq_arr = sLQ_s + slab * (uint32_t)(LQ_SLAB * 4);
    const bool cpass = cmq >= W.min_mapq;
    const uint32_t c1 = c0 + cn;
    uint32_t ob = c0;
    int rp_carry = crel; uint32_t qp_carry = 0;
    if (P.cigar_ckpt) {
        const uint32_t g_first = (c0 >> 5) + 1u, g_last = (c1 - 1u) >> 5;      // checkpoints strictly inside this read
        uint32_t gs = 0;
        for (uint32_t base = g_first; base <= g_last; base += 32) {
            const uint32_t g = base + lane;
            const bool ok = g <= g_last;
            const uint32_t x = ok ? P.cigar_ckpt[g].x : 0u;
            const uint32_t bal = __ballot_sync(FULL, ok && ((long long)crel + (long long)x > 0));   // block starts right of entry 0
            if (bal) { gs = base + (uint32_t)__ffs(bal) - 2u; break; }          // the block before the first such one
            gs = min(g_last, base + 31u);
        }
        if (gs >= g_first) {
            const uint2 ck = P.cigar_ckpt[gs];
            ob = gs << 5;
            rp_carry = (int)min((long long)crel + (long long)ck.x, (long long)WN);
            qp_carry = ck.y;
        }
    }
    uint32_t v = (ob + lane < min(c1, (ob | 31u) + 1u)) ? P.cigar[ob + lane] : 0xfu;
    while (ob < c1) {
        const uint32_t bend = min(c1, (ob | 31u) + 1u);
        const uint32_t op = v & 15u, len = v >> 4;
        // the next block's ops are in flight while this block's qualities are streamed
        const uint32_t nend = min(c1, bend + 32u);
        const uint32_t vn = (bend + lane < nend) ? P.cigar[bend + lane] : 0xfu;
        const uint32_t rl = ((0x18du >> op) & 1u) ? len : 0u, ql = ((0x193u >> op) & 1u) ? len : 0u;
        long long ex_r, tot_r; uint32_t ex_q, tot_q;                   // exclusive prefixes of this lane, block totals
        if (__any_sync(FULL, len >= 2048u)) {
            unsigned long long rs = rl; uint32_t qs = ql;               // 32 ops of < 2^28 bases each: the reference sum needs 33 bits
#pragma unroll 1
            for (int dd = 1; dd < 32; dd <<= 1) {
                const unsigned long long t1 = __shfl_up_sync(FULL, rs, dd); const uint32_t t2 = __shfl_up_sync(FULL, qs, dd);
                if (lane >= dd) { rs += t1; qs += t2; }
            }
            ex_r = (long long)(rs - rl); ex_q = qs - ql;
            tot_r = (long long)__shfl_sync(FULL, rs, 31); tot_q = __shfl_sync(FULL, qs, 31);
        } else {
            uint32_t pk = rl | (ql << 16);                              // every op < 2048 bases: both sums stay below 2^16
#pragma unroll
            for (int dd = 1; dd < 32; dd <<= 1) {
                const uint32_t t = __shfl_up_sync(FULL, pk, dd);
                if (lane >= dd) pk += t;
            }
            ex_r = (long long)((pk & 0xffffu) - rl); ex_q = (pk >> 16) - ql;
            const uint32_t tot = __shfl_sync(FULL, pk, 31);
            tot_r = (long long)(tot & 0xffffu); tot_q = tot >> 16;
        }
        Seg s; bool hs = false;
        const long long my_rel = (long long)rp_carry + ex_r;
        if (cpass && ((0x181u >> op) & 1u) && my_rel < (long long)WN)
            hs = emit_m(W, lq_arr, (int)my_rel, qp_carry + ex_q, len, cq0, clq, s);
        run_segments<BQ_HI>(W, sLQ_s, slab, hs, s, myDesc, sRcp, sMaskLo, sMaskHi, t_low, acc_sum, lane);
        rp_carry = (int)min((long long)rp_carry + tot_r, (long long)WN);   // saturate right of the window
        qp_carry += tot_q;
        if (rp_carry >= (int)W.n_ent) break;                          // rest of the read lies right of the window
        ob = bend; v = vn;
    }
    if (lane == 0) emit_read<WIDE>(W, crel, rp_carry, cmq, acc_mapq);
}

// shared memory: A | B | LQ (KLQ packed-u8 arrays) | masks | first | desc | scan | last | warp stats | next
constexpr size_t SMEM_COUNTER_WORDS = (size_t)WN * 2 + (size_t)LQ_SLAB * KLQ;
// Smallest low-MAPQ count in [0, raw + 1] with (double)low / (double)raw > fraction (callable_profiler.rs:100-101):
// the predicate is monotone in low because IEEE division is monotone.
__device__ __forceinline__ uint32_t first_low(uint32_t raw, double fraction) {
    if (raw == 0) return 0xffffffffu;
    uint32_t lo = 0, hi = raw + 1;
    while (lo < hi) {
        const uint32_t mid = lo + ((hi - lo) >> 1);
        if (__ddiv_rn((double)mid, (double)raw) > fraction) hi = mid; else lo = mid + 1;
    }
    return lo;
}

#ifndef CLB_F_WSTAGE
#define CLB_F_WSTAGE 4880                 // quality bytes one warp of k_pileup_fast stages per sub-batch of <= 32 reads (clb_fast.cuh): 32 x 151 + alignment slack
#endif
#ifndef CLB_PREFETCH_MAX
#define CLB_PREFETCH_MAX (128u << 10)     // bytes of a window's qualities prefetched into L2 at window start
#endif
#ifndef CLB_DCAP
#define CLB_DCAP 1024
#endif
constexpr int DCAP = CLB_DCAP;        // CTA-wide segment pool (descriptors); a 32-read batch adds at most 64
constexpr int BPR = DCAP / 64;        // batches per round
constexpr int CPLX_CAP = BPR * 32;    // long-CIGAR reads queued per round for CTA-wide distribution (a round never holds more reads)
constexpr size_t SMEM_BYTES = SMEM_COUNTER_WORDS * 4 + 2 * 17 * 16 + NFIRST * 4 + NRCP * 4 + (size_t)(NWARPS * 32 + DCAP) * 8 + 64 * 4 + NT
                            + (size_t)NWARPS * N_STATS * 8 + 128 + 2 * CPLX_CAP * 4;
static_assert((size_t)KLQ * LQ_SLAB >= (size_t)WN + 32, "the u32-per-position fallback must fit in the packed low-BQ region");
constexpr size_t SMEM_BYTES_DEEP = SMEM_BYTES + (size_t)WN * 4;      // + the separate low-MAPQ difference array
constexpr size_t WIN_TABLE_BYTES = 2 * 17 * 16 + NFIRST * 4 + NRCP * 4;   // sMaskLo | sMaskHi | sFirst | sRcp, contiguous in shared memory
static_assert(WIN_TABLE_BYTES % 16 == 0, "window tables are copied with 16-byte loads");
static_assert(SMEM_COUNTER_WORDS % 4 == 0 && LQ_SLAB % 4 == 0, "counter region is zeroed with 16-byte stores");

// ---------------------------------------------------------------------------------------------
// What a window leaves for the interval compaction: records of its run starts and one window-table word
// ---------------------------------------------------------------------------------------------
struct IntervalOut { uint32_t start, end; uint8_t state, soft; uint16_t pad; };

// Boundary record: position where a run starts | its state << 32 | soft << 40 (the run merely continues the previous shard's).
__device__ __forceinline__ unsigned long long pack_rec(uint32_t pos, uint32_t state, uint32_t soft) {
    return (unsigned long long)pos | ((unsigned long long)state << 32) | ((unsigned long long)soft << 40);
}
__device__ __forceinline__ IntervalOut unpack_rec(unsigned long long r) {        // end: filled in by k_fill_ends
    IntervalOut iv; iv.start = (uint32_t)r; iv.end = 0; iv.state = (uint8_t)(r >> 32); iv.soft = (uint8_t)((r >> 40) & 1u); iv.pad = 0;
    return iv;
}

// Window table word y: record count | state of entry 0 << 12 | window soft << 16 | state of the last entry << 20.
// "Window soft": the first record was emitted for the window's first position whatever its state (k_pileup_fast has no halo
// entry); the state of entry 0 is only read then.
__device__ __forceinline__ uint32_t pack_win_y(uint32_t count, uint32_t first_state, uint32_t wsoft, uint32_t last_state) {
    return count | (first_state << 12) | (wsoft << 16) | (last_state << 20);
}
__device__ __forceinline__ uint32_t win_count(uint32_t y) { return y & 0xfffu; }
// Records a window contributes to the sorted interval list: its count, minus the window-soft first record when the previous
// window ended in the same state.
__device__ __forceinline__ uint32_t win_drop_first(const uint2 *win_tab, uint32_t w) {
    const uint32_t y = win_tab[w].y;
    if (!((y >> 16) & 1u) || w == 0) return 0u;
    return ((y >> 12) & 15u) == ((win_tab[w - 1].y >> 20) & 15u) ? 1u : 0u;
}
__device__ __forceinline__ uint32_t win_count(uint2 t) { return win_count(t.y); }
__device__ __forceinline__ IntervalOut gather_out(unsigned long long r) { return unpack_rec(r); }

// The depth-run window tables (KParams::run_win_tab, qrun_win_tab) and records: the same compaction reads them.  A
// window-soft first run (k_pileup_fast) is dropped when its depth (raw or QC, the table's kind) equals the previous window's last.
__device__ __forceinline__ uint32_t win_count(uint4 t) { return t.y & 0xffffu; }
__device__ __forceinline__ uint32_t win_drop_first(const uint4 *win_tab, uint32_t w) {
    const uint4 t = win_tab[w];
    if (!((t.y >> 16) & 1u) || w == 0) return 0u;
    return t.z == win_tab[w - 1].w ? 1u : 0u;
}
__device__ __forceinline__ uint2 gather_out(uint2 r) { return r; }

// ---------------------------------------------------------------------------------------------
// Phase C of both pileup kernels (k_pileup_fast, pileup_classify_window): classify the scanned depths, reduce the counters,
// write the run boundaries and the bins.  Thread t holds window entries t * PPT .. t * PPT + PPT - 1.
// ---------------------------------------------------------------------------------------------
using stp_t = typename std::conditional<(PPT > 8), unsigned long long, uint32_t>::type;

// One thread's entries.  Those outside [k_first, k_end) are classified with the rest but do not belong to the window: the
// general kernel's halo (entry 0 of thread 0) and entries past the region end.  Sum: the type of the depth sums (64 bits
// in deep windows, where 32-bit partial sums could overflow).
template <typename Sum>
struct Entries {
    uint32_t ebase, k_first, k_end, vmask;   // vmask: bits [k_first, k_end)
    stp_t stp;                               // 4 bits of state per entry
    uint32_t cnt_pack, covered;              // entries per state (5 bits each), entries with raw depth > 0
    Sum sraw, sqc;
    __device__ __forceinline__ uint32_t state(int k) const { return (uint32_t)(stp >> (4 * k)) & 15u; }
};
template <typename Sum>
__device__ __forceinline__ Entries<Sum> entries_of(uint32_t ebase, uint32_t k_first, uint32_t n_ent) {
    Entries<Sum> e;
    e.ebase = ebase; e.k_first = k_first;
    e.k_end = n_ent > ebase ? min((uint32_t)PPT, n_ent - ebase) : 0u;
    e.vmask = ((1u << e.k_end) - 1u) & ~((1u << k_first) - 1u);          // k_end >= k_first: a window has >= 2 entries
    e.stp = 0; e.cnt_pack = 0; e.covered = 0; e.sraw = 0; e.sqc = 0;
    return e;
}

// The options' depth thresholds, read once per window
struct StateLimits { uint32_t min_depth_for_low_mapq, min_depth, max_depth; };
__device__ __forceinline__ StateLimits state_limits(const KParams &P) {
    return StateLimits{P.min_depth_for_low_mapq, P.min_depth, P.max_depth ? P.max_depth : 0xffffffffu};   // max_depth == 0 disables EXCESSIVE_COVERAGE
}

// State of entry k (callable_profiler.rs:89-120).  fst: the smallest low-MAPQ depth that makes raw depth POOR_MAPPING_QUALITY.
template <typename Sum>
__device__ __forceinline__ void classify_entry(Entries<Sum> &e, int k, uint32_t raw, uint32_t low, uint32_t qc, uint32_t fst, uint32_t ref_n,
                                               const StateLimits &lim) {
    const bool is_low = raw >= lim.min_depth_for_low_mapq && low >= fst;
    uint32_t s = qc > lim.max_depth ? ST_EXCESSIVE : ST_CALLABLE;
    s = qc < lim.min_depth ? ST_LOW_COVERAGE : s;
    s = is_low ? ST_POOR_MAPQ : s;
    s = raw == 0 ? ST_NO_COVERAGE : s;
    s = ref_n ? ST_REF_N : s;
    e.stp |= (stp_t)s << (4 * k);
    e.cnt_pack += 1u << (5 * s);
    e.covered += raw > 0 ? 1u : 0u;
    e.sraw += raw; e.sqc += qc;
}

// Depth histograms (HIST instantiations; DESIGN.md §4).  Each CTA counts into a table of DH_TAB u32 bins per histogram in
// shared memory (raw at s_tab, qc at s_tab + 4 * DH_TAB), zeroed at the start of phase C, and flushes it after the
// reduce_stats barrier into its global slot copy; a clamped depth past the table (general and deep kernels only) goes to the
// slot copy directly.  A thread merges runs of equal depth over its entries in registers first (depth changes at read ends
// only, so at 30x a thread's 8 entries hold two or three runs): one predicated shared atomic per run instead of per entry.
#ifndef CLB_DH_SLOTS
#define CLB_DH_SLOTS 16
#endif
constexpr int DH_SLOTS = CLB_DH_SLOTS;   // global copies of the histograms (blockIdx.x % DH_SLOTS): spreads the flush atomics
constexpr int DH_TAB = 256;              // shared bins per histogram: every depth the fast kernel can see (raw <= 254)
struct DepthHist {
    uint32_t s_tab, nm1;                 // shared table, n - 1
    unsigned long long *g;               // this CTA's slot copy: [raw n][qc n]
    uint32_t rd, rc, qd, qn;             // open runs: (depth, entries) of raw and qc
};
__device__ __forceinline__ DepthHist depth_hist_of(uint32_t s_tab, const KParams &P) {
    return DepthHist{s_tab, P.dh_n - 1u, P.dhist + (size_t)(blockIdx.x % DH_SLOTS) * 2u * P.dh_n, 0u, 0u, 0u, 0u};
}
// TAB_ONLY: the caller's depths never exceed DH_TAB - 1 (k_pileup_fast's depth proof)
template <bool TAB_ONLY>
__device__ __forceinline__ void depth_hist_add(const DepthHist &h, uint32_t which, uint32_t d, uint32_t cnt) {
    if (TAB_ONLY || d < (uint32_t)DH_TAB) red_shared_nz(h.s_tab + 4u * ((uint32_t)DH_TAB * which + d), cnt);
    else if (cnt) atomicAdd(h.g + (size_t)which * (h.nm1 + 1u) + d, (unsigned long long)cnt);
}
// Entry k of the classification: counts when it is one of the window's own entries (vmask: not the general kernel's halo,
// not past the region end) and not REF_N, at depth min(depth, n - 1).
template <bool TAB_ONLY, typename Sum>
__device__ __forceinline__ void count_depth(DepthHist &h, const Entries<Sum> &e, int k, uint32_t raw, uint32_t qc) {
    const uint32_t one = (((e.vmask >> k) & 1u) && e.state(k) != ST_REF_N) ? 1u : 0u;
    const uint32_t dr = min(raw, h.nm1), dq = min(qc, h.nm1);
    const bool br = dr != h.rd, bq = dq != h.qd;
    depth_hist_add<TAB_ONLY>(h, 0u, h.rd, br ? h.rc : 0u);          // a run ends: add it
    depth_hist_add<TAB_ONLY>(h, 1u, h.qd, bq ? h.qn : 0u);
    h.rc = (br ? 0u : h.rc) + one; h.rd = dr;
    h.qn = (bq ? 0u : h.qn) + one; h.qd = dq;
}
template <bool TAB_ONLY>
__device__ __forceinline__ void close_depth_runs(DepthHist &h) {
    depth_hist_add<TAB_ONLY>(h, 0u, h.rd, h.rc);
    depth_hist_add<TAB_ONLY>(h, 1u, h.qd, h.qn);
}
// Before the barrier that precedes the first count_depth; the table must be dead (no other phase uses it any more).
__device__ __forceinline__ void zero_depth_table(uint32_t *tab) {
    for (int i = threadIdx.x; i < 2 * DH_TAB; i += NT) tab[i] = 0u;
}
// After a barrier that follows every close_depth_runs: the table's non-zero bins to the CTA's slot copy.
__device__ __forceinline__ void flush_depth_table(const DepthHist &h, const uint32_t *tab) {
    for (int i = threadIdx.x; i < 2 * DH_TAB; i += NT) {
        const uint32_t which = (uint32_t)i / DH_TAB, d = (uint32_t)i % DH_TAB, v = tab[i];
        if (v && d <= h.nm1) atomicAdd(h.g + (size_t)which * (h.nm1 + 1u) + d, (unsigned long long)v);
    }
}

// Entries outside [k_first, k_end) were counted as states: take them out again.  Then publish what the boundary pass reads
// from other threads: the state of this thread's last entry and that of the window's last position.
template <typename Sum>
__device__ __forceinline__ void close_entries(Entries<Sum> &e, uint32_t n_ent, uint8_t *sLast, uint32_t *sScan) {
    uint32_t inv = ~e.vmask & ((1u << PPT) - 1u);
    while (inv) {
        const int k = __ffs(inv) - 1; inv &= inv - 1;
        e.cnt_pack -= 1u << (5 * e.state(k));
    }
    sLast[threadIdx.x] = (uint8_t)e.state(PPT - 1);
    if (e.k_end > e.k_first && e.ebase + e.k_end == n_ent) sScan[3 * NWARPS + 1] = e.state(e.k_end - 1);
}

// Per-base dump for the parity tests (own instantiation).  o0: offset of entry 0 from the region start; entry(k) = (raw, qc, low).
template <bool DBG, typename Sum, typename Entry>
__device__ __forceinline__ void dbg_dump(const Entries<Sum> &e, uint32_t o0, Entry entry, const KParams &P) {
    if (DBG && P.dbg_raw) {
#pragma unroll
        for (int k = 0; k < PPT; k++) if ((e.vmask >> k) & 1u) {
            const uint3 v = entry(k);
            const uint32_t o = o0 + e.ebase + k;
            P.dbg_raw[o] = v.x; P.dbg_qc[o] = v.y; P.dbg_low[o] = v.z; P.dbg_state[o] = (uint8_t)e.state(k);
        }
    }
}

__device__ __forceinline__ uint32_t warp_sum(uint32_t v) { return __reduce_add_sync(FULL, v); }
__device__ __forceinline__ unsigned long long warp_sum(unsigned long long v) {
#pragma unroll
    for (int dd = 16; dd > 0; dd >>= 1) v += __shfl_xor_sync(FULL, v, dd);
    return v;
}

// Depth tiles (TILES instantiations; DESIGN.md §4).  Per tile: the own positions that are not REF_N (territory), the
// CALLABLE ones, and the raw and QC depth sums over the former.  A thread's entries cross at most one tile boundary and a
// warp's 256 entries touch at most two tiles (tile_len >= 256): each warp sums into its two tiles and parks them in its
// slot; after the reduce_stats barrier the CTA adds the slots up for the at most TL_MAX tiles of the window and flushes
// them with one global atomic per non-zero (tile, counter).  The slots sit beside the depth table (both may be on).
constexpr int TL_MAX = 9;                                   // tiles one window can touch: 2047 positions, tiles of >= 256
constexpr int TL_SLOT_BYTES = NWARPS * (8 * 8 + 4);         // per warp [2 tiles][4 counters] u64, then per warp its first tile (u32)
// Depth thresholds (THRESH instantiations, always with TILES; DESIGN.md §4): per tile and threshold j, the tile's own
// positions that are not REF_N with raw (QC) depth >= thr[j].  A depth maps to a word of unary nibbles, nibble j = (depth >=
// thr[j]); a thread adds its entries' words per tile and kind (at most 8 per nibble: no carry) and the warp sums them as
// 16-bit pairs of nibbles j and j + 4 (at most 256 per half), four REDUX per tile and kind.  Nibbles j >= n_thr are never
// flushed.  The words of depths below TH_TAB come from a shared table filled once per window.
constexpr int TH_TAB = 256;                                 // table entries: every depth the fast kernel can see (raw <= 254)
constexpr int TH_SLOT_BYTES = NWARPS * 2 * 2 * 16;          // per warp [2 tiles][raw, qc] uint4 of 16-bit pairs
static_assert(4 * TL_MAX + 2 * TH_MAX * TL_MAX <= NT, "one flush thread per tile counter and per tile threshold count");
__device__ __forceinline__ uint32_t thresh_nibbles(uint32_t d, const KParams &P) {
    uint32_t v = 0u;
#pragma unroll
    for (int j = 0; j < TH_MAX; j++) v += d >= P.thr[j] ? 1u << (4 * j) : 0u;
    return v;
}
// Before the barrier that precedes count_tiles; the table must be dead (no other phase uses it any more).
__device__ __forceinline__ void fill_thresh_table(uint32_t *tab, const KParams &P) {
    for (int i = threadIdx.x; i < TH_TAB; i += NT) tab[i] = thresh_nibbles((uint32_t)i, P);
}
// The warp's sums of a nibble word as 16-bit pairs: .x = (nibble 0, nibble 4), .y = (1, 5), .z = (2, 6), .w = (3, 7)
__device__ __forceinline__ uint4 warp_sum_nibbles(uint32_t v) {
    const uint32_t m = 0x000f000fu;
    return make_uint4(warp_sum(v & m), warp_sum((v >> 4) & m), warp_sum((v >> 8) & m), warp_sum((v >> 12) & m));
}

// After close_entries and the general kernel's halo correction: cnt_pack, sraw and sqc cover the own entries only (entries
// past the region end carry no depth).  pos0: position of entry 0; depth(k) = (raw, qc) of entry k.  THRESH: also the
// threshold counts, from sThTab (filled by fill_thresh_table) for depths below TH_TAB (TAB_ONLY: the caller's depths always
// are), into sThSlot (TH_SLOT_BYTES, 16-byte aligned).
template <bool THRESH = false, bool TAB_ONLY = false, typename Sum, typename Depth>
__device__ __forceinline__ void count_tiles(const Entries<Sum> &e, uint32_t pos0, uint32_t nbits, Depth depth, unsigned long long *sTileSum,
                                            uint32_t *sTileFirst, const KParams &P, const uint32_t *sThTab = nullptr,
                                            uint32_t *sThSlot = nullptr) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t L = P.tile_len;
    const uint32_t p = pos0 + e.ebase + e.k_first;                        // the thread's first own entry (never the halo)
    const uint32_t t = p / L;
    const uint32_t split = e.k_first + min(L - (p - t * L), (uint32_t)PPT);   // entries below split lie in tile t, the rest in t + 1
    const uint32_t own = e.vmask & ~nbits;                                // own entries that are not REF_N
    uint32_t ter0 = __popc(own), cal0 = (e.cnt_pack >> (5 * ST_CALLABLE)) & 31u, ter1 = 0u, cal1 = 0u;
    Sum raw0 = e.sraw, qc0 = e.sqc, raw1 = 0, qc1 = 0;
    if (own != e.vmask || split < e.k_end) {                              // REF_N depth in the sums, or a tile boundary (rare)
        ter0 = cal0 = 0u; raw0 = qc0 = 0;
#pragma unroll
        for (int k = 0; k < PPT; k++) {
            const uint2 d = depth(k);
            const uint32_t o = (own >> k) & 1u, c = o && e.state(k) == ST_CALLABLE ? 1u : 0u;
            const Sum r = o ? (Sum)d.x : (Sum)0, q = o ? (Sum)d.y : (Sum)0;
            if ((uint32_t)k < split) { ter0 += o; cal0 += c; raw0 += r; qc0 += q; }
            else { ter1 += o; cal1 += c; raw1 += r; qc1 += q; }
        }
    }
    uint32_t gr0 = 0u, gq0 = 0u, gr1 = 0u, gq1 = 0u;                      // THRESH: raw / QC nibble words of tiles t and t + 1
    if constexpr (THRESH) {
        const uint32_t in0 = own & ((1u << split) - 1u);                  // own entries in tile t
        const auto add = [&](auto tab_tag) {
#pragma unroll
            for (int k = 0; k < PPT; k++) {
                const uint2 d = depth(k);
                const uint32_t r = decltype(tab_tag)::value ? sThTab[d.x] : thresh_nibbles(d.x, P);
                const uint32_t q = decltype(tab_tag)::value ? sThTab[d.y] : thresh_nibbles(d.y, P);
                if ((in0 >> k) & 1u) { gr0 += r; gq0 += q; }
                else if ((own >> k) & 1u) { gr1 += r; gq1 += q; }
            }
        };
        if constexpr (TAB_ONLY) {
            add(std::true_type{});
        } else {
            uint32_t deepest = 0u;                                        // an upper bound of the thread's depths
#pragma unroll
            for (int k = 0; k < PPT; k++) { const uint2 d = depth(k); deepest |= d.x | d.y; }
            if (deepest < (uint32_t)TH_TAB) add(std::true_type{}); else add(std::false_type{});
        }
    }
    const uint32_t T = __shfl_sync(FULL, t, 0);                           // the warp's first tile
    if (t != T) {                                                         // then nothing reached t + 1
        ter1 = ter0; cal1 = cal0; raw1 = raw0; qc1 = qc0; ter0 = cal0 = 0u; raw0 = qc0 = 0;
        if constexpr (THRESH) { gr1 = gr0; gq1 = gq0; gr0 = gq0 = 0u; }
    }
    const uint32_t s0 = warp_sum(ter0), s1 = warp_sum(cal0);
    const Sum s2 = warp_sum(raw0), s3 = warp_sum(qc0);
    uint32_t u0 = 0u, u1 = 0u; Sum u2 = 0, u3 = 0;
    if (__any_sync(FULL, ter1 != 0u)) { u0 = warp_sum(ter1); u1 = warp_sum(cal1); u2 = warp_sum(raw1); u3 = warp_sum(qc1); }   // warp-uniform
    if (lane == 0) {
        unsigned long long *ws = sTileSum + warp * 8;
        ws[0] = s0; ws[1] = s1; ws[2] = s2; ws[3] = s3; ws[4] = u0; ws[5] = u1; ws[6] = u2; ws[7] = u3;
        sTileFirst[warp] = T;
    }
    if constexpr (THRESH) {
        const uint4 r0 = warp_sum_nibbles(gr0), q0 = warp_sum_nibbles(gq0);
        uint4 r1 = make_uint4(0u, 0u, 0u, 0u), q1 = r1;
        if (__any_sync(FULL, ter1 != 0u)) { r1 = warp_sum_nibbles(gr1); q1 = warp_sum_nibbles(gq1); }   // warp-uniform
        if (lane == 0) {
            uint4 *ts = reinterpret_cast<uint4 *>(sThSlot) + warp * 4;
            ts[0] = r0; ts[1] = q0; ts[2] = r1; ts[3] = q1;
        }
    }}
// Thread 4 * TL_MAX + (kind * TH_MAX + j) * TL_MAX + i adds threshold j's raw (kind 0) or QC (kind 1) count of the window's
// tile i; flush_tiles calls it.
__device__ __forceinline__ void flush_thresholds(const uint32_t *sThSlot, const uint32_t *sTileFirst, const KParams &P) {
    const uint32_t i = threadIdx.x - 4u * TL_MAX;
    const uint32_t kind = i / (TH_MAX * TL_MAX), j = i / TL_MAX % TH_MAX, ti = i % TL_MAX, t0 = sTileFirst[0];
    if (kind >= 2u || j >= P.n_thr) return;
    const uint32_t word = kind * 4u + (j & 3u), shift = 16u * (j >> 2);   // [tile][kind][pair word]; nibble j in half j >> 2
    uint32_t s = 0u;
#pragma unroll
    for (int w = 0; w < NWARPS; w++) {
        const uint32_t d = sTileFirst[w] - t0;
        if (d == ti) s += (sThSlot[w * 16 + word] >> shift) & 0xffffu;
        if (d + 1u == ti) s += (sThSlot[w * 16 + 8 + word] >> shift) & 0xffffu;
    }
    if (s && t0 + ti < P.n_tiles) atomicAdd(P.tiles + (size_t)(4u + kind * P.n_thr + j) * P.n_tiles + t0 + ti, (unsigned long long)s);
}
// After a barrier that follows every count_tiles: thread c * TL_MAX + j adds counter c of the window's tile j; THRESH: the
// next 2 * TH_MAX * TL_MAX threads add the threshold counts.
template <bool THRESH = false>
__device__ __forceinline__ void flush_tiles(const unsigned long long *sTileSum, const uint32_t *sTileFirst, const KParams &P,
                                            const uint32_t *sThSlot = nullptr) {
    const uint32_t i = threadIdx.x;
    if (i >= 4u * TL_MAX) {
        if constexpr (THRESH) flush_thresholds(sThSlot, sTileFirst, P);
        return;
    }
    const uint32_t c = i / TL_MAX, j = i % TL_MAX, t0 = sTileFirst[0];
    unsigned long long s = 0;
#pragma unroll
    for (int w = 0; w < NWARPS; w++) {
        const uint32_t d = sTileFirst[w] - t0;
        if (d == j) s += sTileSum[w * 8 + c];
        if (d + 1u == j) s += sTileSum[w * 8 + 4 + c];
    }
    if (s && t0 + j < P.n_tiles) atomicAdd(P.tiles + (size_t)c * P.n_tiles + t0 + j, s);
}

// Counters: per-warp sums in plain stores (no 64-bit shared atomics), summed after a barrier into one global atomic per
// counter.  acc_sum / acc_mapq: the thread's base-quality and MAPQ sums (MapqSum: 64 bits unless the window's sum fits 32).
template <typename Sum, typename MapqSum>
__device__ __forceinline__ void reduce_stats(const Entries<Sum> &e, uint32_t acc_sum, MapqSum acc_mapq, unsigned long long *sWStats,
                                             const KParams &P) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint32_t v[7];
#pragma unroll
    for (int s = 0; s < 6; s++) v[s] = (e.cnt_pack >> (5 * s)) & 31u;
    v[6] = e.covered;
#pragma unroll
    for (int i = 0; i < 7; i++) v[i] = __reduce_add_sync(FULL, v[i]);
    const Sum sraw = warp_sum(e.sraw), sqc = warp_sum(e.sqc), sbq = warp_sum((Sum)acc_sum);
    const MapqSum smq = warp_sum(acc_mapq);
    if (lane == 0) {
        unsigned long long *ws = sWStats + warp * N_STATS;
#pragma unroll
        for (int s = 0; s < 6; s++) ws[S_COUNT0 + s] = v[s];
        ws[S_COVERED] = v[6]; ws[S_SUMCOV] = sraw; ws[S_SUMBQ] = sbq; ws[S_QBASES] = sqc;
        ws[S_RESERVED] = 0; ws[S_SUMMAPQ] = smq;
    }
    __syncthreads();
    if (tid < N_STATS) {
        unsigned long long t = 0;
#pragma unroll
        for (int j = 0; j < NWARPS; j++) t += sWStats[j * N_STATS + tid];
        if (t) atomicAdd(&P.stats[tid * STAT_STRIDE], t);
    }
}

// Depth runs (RUNS instantiations; DESIGN.md §4).  Entry k starts a run iff its raw depth differs from entry k - 1's.  A
// thread takes the previous thread's last raw depth by shuffle within the warp and, for lane 0, from the previous warp's
// word in sRunLast.  raw(k): raw depth of entry k.  QC depth runs (QRUNS) are the same calls with the QC depth, their own
// per-warp words and their own sScan words.
// sScan words: 3 * NWARPS + 2 / + 3 (window's last raw depth, run base), + 4 / + 5 (the same for QC runs), 5 * NWARPS + warp
// (per-warp QC run counts when both kinds are on)
static_assert(3 * NWARPS + 6 <= 4 * NWARPS && 6 * NWARPS <= 64, "sScan words of the depth runs");
// Before reduce_stats' barrier: lane 31 parks the warp's last depth, the thread holding the window's last position that
// position's depth in *sWinLast.
template <typename Sum, typename Raw>
__device__ __forceinline__ void publish_run_depth(const Entries<Sum> &e, uint32_t n_ent, Raw raw, uint32_t *sRunLast, uint32_t *sWinLast) {
    if ((threadIdx.x & 31) == 31) sRunLast[threadIdx.x >> 5] = raw(PPT - 1);
    if (e.k_end > e.k_first && e.ebase + e.k_end == n_ent) {
        uint32_t last = 0;
#pragma unroll
        for (int k = 0; k < PPT; k++) last = (uint32_t)k + 1u == e.k_end ? raw(k) : last;
        *sWinLast = last;
    }
}
// After that barrier: the thread's own entries that start a run, plus those in force.  Thread 0's entry 0 always starts one
// (k_pileup_fast has no halo; the general kernel's entry 0 is the halo, outside vmask).
template <typename Sum, typename Raw>
__device__ __forceinline__ uint32_t run_starts(const Entries<Sum> &e, Raw raw, uint32_t force, const uint32_t *sRunLast) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t up = __shfl_up_sync(FULL, raw(PPT - 1), 1);
    uint32_t prev = lane > 0 ? up : warp > 0 ? sRunLast[warp - 1] : 0xffffffffu;
    uint32_t m = 0;
#pragma unroll
    for (int k = 0; k < PPT; k++) { const uint32_t d = raw(k); m |= (d != prev ? 1u : 0u) << k; prev = d; }
    return (m | force) & e.vmask;
}

// One depth-run stream of write_records (thread 0): reserve the window's cnt records from cursor and describe them in
// win_tab[w] = (first record, count | window soft << 16, depth of the first own entry, of the last); the first record's
// index goes to *sBase.
__device__ __forceinline__ void reserve_runs(uint32_t *cursor, uint4 *win_tab, uint32_t w, uint32_t cnt, uint32_t win_soft, uint32_t first,
                                             uint32_t last, uint32_t *sBase) {
    const uint32_t rbase = atomicAdd(cursor, cnt);
    *sBase = rbase;
    win_tab[w] = make_uint4(rbase, cnt | (win_soft << 16), first, last);
}
// ... and every thread: the starts in mask, (position, depth(k)) each, from record o on.  p0: position of entry 0.
template <typename Depth>
__device__ __forceinline__ void write_runs(uint32_t mask, Depth depth, uint32_t o, uint32_t p0, uint2 *rec, uint32_t cap) {
#pragma unroll
    for (int k = 0; k < PPT; k++) {                                       // unrolled: depth(k) stays in registers
        if ((mask >> k) & 1u) {
            if (o < cap) rec[o] = make_uint2(p0 + k, depth(k));
            o++;
        }
    }
}

// Run boundaries -> records.  Entry k starts a run iff its state differs from entry k - 1's; thread 0's entry 0 always does.
// The entries in force start a record regardless; those in soft (a subset of force) that merely continue a run are flagged
// soft.  pos0: position of entry 0; win_soft: see pack_win_y.  RUNS / QRUNS: the depth-run starts in rmask / qmask go to the
// raw / QC run records in the same scan; raw(k) / qc(k) is entry k's raw / QC depth.  With one run kind on, its count rides
// in the scan word (state count | run count << 16: both <= 2047 per window); with both, the QC count has a second word.
template <bool RUNS, bool QRUNS, typename Sum, typename Raw, typename Qc>
__device__ __forceinline__ void write_records(const Entries<Sum> &e, uint32_t pos0, uint32_t force, uint32_t soft, uint32_t win_soft,
                                              const uint8_t *sLast, uint32_t *sScan, uint32_t w, const KParams &P, uint32_t rmask,
                                              Raw raw, uint32_t qmask, Qc qc) {
    constexpr bool ANY = RUNS || QRUNS, BOTH = RUNS && QRUNS;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint32_t bmask, softmask;
    {
        const uint32_t prev_last = tid > 0 ? sLast[tid - 1] : 0xfu;       // no state is 15
        const stp_t shifted = (e.stp << 4) | (stp_t)prev_last;            // state of entry k-1 in nibble k
        stp_t diff = e.stp ^ shifted;                                      // non-zero nibble <=> boundary
        diff |= diff >> 1; diff |= diff >> 2;                              // bit 4k collects the nibble
        bmask = 0;
#pragma unroll
        for (int k = 0; k < PPT; k++) bmask |= ((uint32_t)(diff >> (4 * k)) & 1u) << k;
        softmask = soft & ~bmask;
        bmask = (bmask | force) & e.vmask;
    }
    const uint32_t nb = ANY ? __popc(bmask) | (__popc(RUNS ? rmask : qmask) << 16) : __popc(bmask);
    const uint32_t nq = BOTH ? __popc(qmask) : 0u;
    uint32_t inb = nb, inq = nq;
#pragma unroll
    for (int dd = 1; dd < 32; dd <<= 1) {
        const uint32_t t = __shfl_up_sync(FULL, inb, dd);
        if (BOTH) { const uint32_t tq = __shfl_up_sync(FULL, inq, dd); if (lane >= dd) inq += tq; }
        if (lane >= dd) inb += t;
    }
    if (lane == 31) { sScan[2 * NWARPS + warp] = inb; if (BOTH) sScan[5 * NWARPS + warp] = inq; }
    __syncthreads();
    const uint32_t wt = lane < NWARPS ? sScan[2 * NWARPS + lane] : 0u;             // lane j: boundaries in warp j
    uint32_t off = inb - nb + __reduce_add_sync(FULL, lane < warp ? wt : 0u), total = __reduce_add_sync(FULL, wt);
    const uint32_t roff = off >> 16, rtotal = total >> 16;                // the run kind in the high half
    if (ANY) { off &= 0xffffu; total &= 0xffffu; }
    uint32_t qoff = roff, qtotal = rtotal;                                 // QC runs: the high half, or the second word
    if (BOTH) {
        const uint32_t wq = lane < NWARPS ? sScan[5 * NWARPS + lane] : 0u;
        qoff = inq - nq + __reduce_add_sync(FULL, lane < warp ? wq : 0u); qtotal = __reduce_add_sync(FULL, wq);
    }
    if (tid == 0) {
        const uint32_t base = atomicAdd(P.rec_cursor, total);                 // total may be 0 (general kernel): base is not read then
        sScan[3 * NWARPS] = base;
        P.win_tab[w] = make_uint2(base, pack_win_y(total, e.state(0), win_soft, sScan[3 * NWARPS + 1]));
        if ((unsigned long long)base + total > P.rec_cap) atomicOr(P.err, ERR_REC_OVERFLOW);
        if (RUNS) reserve_runs(P.run_cursor, P.run_win_tab, w, rtotal, win_soft, raw(0), sScan[3 * NWARPS + 2], sScan + 3 * NWARPS + 3);
        if (QRUNS) reserve_runs(P.qrun_cursor, P.qrun_win_tab, w, qtotal, win_soft, qc(0), sScan[3 * NWARPS + 4], sScan + 3 * NWARPS + 5);
    }
    __syncthreads();
    uint32_t o = sScan[3 * NWARPS] + off;
    uint32_t m = bmask;
    while (m) {
        const int k = __ffs(m) - 1; m &= m - 1;
        if (o < P.rec_cap) P.rec[o] = pack_rec(pos0 + e.ebase + k, e.state(k), (softmask >> k) & 1u);
        o++;
    }
    if (RUNS) write_runs(rmask, raw, sScan[3 * NWARPS + 3] + roff, pos0 + e.ebase, P.run_rec, P.run_cap);
    if (QRUNS) write_runs(qmask, qc, sScan[3 * NWARPS + 5] + qoff, pos0 + e.ebase, P.qrun_rec, P.qrun_cap);
}

// Bins: positions of CALLABLE / POOR_MAPPING_QUALITY / REF_N per stride-sized bin.  pos0: position of entry 0; e_first: the
// window's first own entry (1 with a halo, else 0); fb, nbe: the window's first bin and the entry where the next bin starts.
template <typename Sum>
__device__ __forceinline__ void add_bins(const Entries<Sum> &e, uint32_t pos0, uint32_t e_first, uint32_t n_ent, uint32_t fb, uint32_t nbe,
                                         const KParams &P) {
    if (!P.n_bins) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t c_call = (e.cnt_pack >> (5 * ST_CALLABLE)) & 31u, c_poor = (e.cnt_pack >> (5 * ST_POOR_MAPQ)) & 31u, c_refn = e.cnt_pack & 31u;
    const uint32_t we0 = max(e_first, (uint32_t)(warp * 32 * PPT)), we1 = min(n_ent, (uint32_t)((warp + 1) * 32 * PPT));
    if (we1 <= we0) return;                                                // warp-uniform
    uint32_t wbin0, wbin1;
    if (we1 <= nbe) { wbin0 = wbin1 = fb; }
    else if (we0 >= nbe && we1 - nbe <= P.stride) { wbin0 = wbin1 = fb + 1; }
    else { wbin0 = (pos0 + we0) / P.stride; wbin1 = (pos0 + we1 - 1) / P.stride; }
    if (wbin0 == wbin1) {                                                  // whole warp inside one bin (the common case: stride >> 256)
        const uint32_t s0 = __reduce_add_sync(FULL, c_call), s1 = __reduce_add_sync(FULL, c_poor), s2 = __reduce_add_sync(FULL, c_refn);
        if (lane == 0) {
            if (s0) atomicAdd(&P.bins[wbin0], (unsigned long long)s0);
            if (s1) atomicAdd(&P.bins[P.n_bins + wbin0], (unsigned long long)s1);
            if (s2) atomicAdd(&P.bins[2 * P.n_bins + wbin0], (unsigned long long)s2);
        }
    } else if (e.k_end > e.k_first) {
        const uint32_t tb0 = (pos0 + e.ebase + e.k_first) / P.stride, tb1 = (pos0 + e.ebase + e.k_end - 1) / P.stride;
        if (tb0 == tb1) {
            if (c_call) atomicAdd(&P.bins[tb0], (unsigned long long)c_call);
            if (c_poor) atomicAdd(&P.bins[P.n_bins + tb0], (unsigned long long)c_poor);
            if (c_refn) atomicAdd(&P.bins[2 * P.n_bins + tb0], (unsigned long long)c_refn);
        } else {
#pragma unroll 1                                                // rare (a thread's entries straddle two bins): keep it small
            for (uint32_t k = e.k_first; k < e.k_end; k++) {
                const uint32_t bi = (pos0 + e.ebase + k) / P.stride;
                const uint32_t s = e.state(k);
                if (s == ST_CALLABLE) atomicAdd(&P.bins[bi], 1ull);
                else if (s == ST_POOR_MAPQ) atomicAdd(&P.bins[P.n_bins + bi], 1ull);
                else if (s == ST_REF_N) atomicAdd(&P.bins[2 * P.n_bins + bi], 1ull);
            }
        }
    }
}

// One window.  WIDE = false packs the raw and low-MAPQ depths as 16 + 16 bits (windows with <= 65535 candidate reads, i.e.
// practically all of them); WIDE = true keeps them in two 32-bit arrays and is only instantiated by k_pileup_classify_deep.
// FEAT: also count the depth histograms and / or the depth tiles (the segment pool, dead in phase C, holds their shared
// tables).
template <bool BQ_HI, bool WIDE, bool DBG, unsigned FEAT>
__device__ __forceinline__ void pileup_classify_window(const KParams &P, const uint32_t w) {
    constexpr bool HIST = (FEAT & FEAT_HIST) != 0, TILES = (FEAT & FEAT_TILES) != 0, RUNS = (FEAT & FEAT_RUNS) != 0;
    constexpr bool THRESH = (FEAT & FEAT_THRESH) != 0, QRUNS = (FEAT & FEAT_QRUNS) != 0;
    static_assert(!THRESH || TILES, "depth thresholds are counted per depth tile");
    extern __shared__ __align__(16) uint8_t smem_raw[];
    uint32_t *sA = reinterpret_cast<uint32_t *>(smem_raw);
    uint32_t *sB = sA + WN;
    uint32_t *sLQ = sB + WN;
    uint4 *sMaskLo = reinterpret_cast<uint4 *>(sLQ + LQ_SLAB * KLQ);
    uint4 *sMaskHi = sMaskLo + 17;
    uint32_t *sFirst = reinterpret_cast<uint32_t *>(sMaskHi + 17);
    uint32_t *sRcp = sFirst + NFIRST;
    uint2 *sDesc = reinterpret_cast<uint2 *>(sRcp + NRCP);
    uint2 *sPool = sDesc + NWARPS * 32;
    uint32_t *sScan = reinterpret_cast<uint32_t *>(sPool + DCAP);
    uint8_t *sLast = reinterpret_cast<uint8_t *>(sScan + 64);
    unsigned long long *sWStats = reinterpret_cast<unsigned long long *>(sLast + NT);
    uint32_t *sCtl = reinterpret_cast<uint32_t *>(sWStats + NWARPS * N_STATS);   // [parity][next batch, pool count, pool max chunks]

    uint32_t *sLowD = reinterpret_cast<uint32_t *>(smem_raw + SMEM_BYTES);       // WIDE only
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    CLB_STAMP(0);

    Win W;
    W.wb = (long long)P.region_start + (long long)w * WREAL - 1;
    W.wend = min(W.wb + WN, (long long)P.region_end);
    W.qual = P.qual; W.qual_bytes = P.qual_bytes; W.sA = smem_addr(sA); W.sB = smem_addr(sB); W.sL = WIDE ? smem_addr(sLowD) : 0u;
    W.min_bq = P.min_bq; W.min_mapq = P.min_mapq; W.max_low_mapq = P.max_low_mapq;
    const uint32_t n_ent = (uint32_t)(W.wend - W.wb);      // entries in use, >= 2
    W.n_ent = n_ent;
    const uint4 wr = P.win_rec[3 * (size_t)w];
    const ulonglong2 wq = *reinterpret_cast<const ulonglong2 *>(P.win_rec + 3 * (size_t)w + 1);
    const uint32_t r_lo = wr.x, r_hi = wr.y;
    const uint32_t n_batches = (r_hi - r_lo + 31u) >> 5;
    const uint32_t n_lq = (n_batches + BPA - 1) / BPA;     // packed arrays needed
    W.lq_packed = n_lq <= (uint32_t)KLQ;
    W.qbase = 0;
    if (r_hi > r_lo) {
        W.qbase = wq.x;
        if (wq.y - W.qbase > 0xfffffff0ull) {
            // 32-bit quality offsets cannot represent this window
            if (tid == 0) { atomicOr(P.err, ERR_QUAL_SPAN); P.win_tab[w] = make_uint2(0, 0); }
            return;
        }
        if (!WIDE && r_hi - r_lo > 65535u) {
            // the 16-bit depth fields could overflow: queue the window for the deep pass
            if (tid == 0) { P.deep_list[atomicAdd(P.deep_count, 1u)] = w; P.win_tab[w] = make_uint2(0, 0); }
            return;
        }
    }
    // The window's qualities are one contiguous byte range that phase B streams after the CIGAR walk: start pulling it
    // into L2 now (one bulk prefetch: no registers, no shared memory).  Prefetching the inputs of the window one wave
    // of CTAs further on as well was measured and lost 3-6 %.
    if (tid == 0) l2_prefetch(P.qual, wq.x, wq.y, CLB_PREFETCH_MAX);

    {
        // zero the difference arrays and only the low-BQ slabs this window will use
        uint4 *z = reinterpret_cast<uint4 *>(sA);
        const int nz = (int)((2 * WN + (W.lq_packed ? n_lq : (uint32_t)KLQ) * LQ_SLAB) / 4);
        for (int i = tid; i < nz; i += NT) z[i] = make_uint4(0, 0, 0, 0);
        if (WIDE) for (int i = tid; i < WN; i += NT) sLowD[i] = 0u;
    }
    {
        // byte masks, first_tab[0..NFIRST) and the reciprocal table: built once per context (k_window_tables), copied here
        const uint4 *src = reinterpret_cast<const uint4 *>(P.win_tables);
        uint4 *dst = sMaskLo;
        for (int i = tid; i < (int)(WIN_TABLE_BYTES / 16); i += NT) dst[i] = src[i];
    }
    if (tid < 6) sCtl[tid] = 0;
    if (tid >= 16 && tid < 20) sCtl[tid] = 0;                // [16 + 2 * parity]: queued long reads, next to expand
    uint32_t *sCplx = sCtl + 32;                            // [parity][CPLX_CAP] read indices
    if (tid == 0) {                                          // runtime divisions once per CTA instead of once per thread
        const uint32_t nr = (n_batches + BPR - 1) / BPR;
        sCtl[8] = nr; sCtl[9] = nr ? (n_batches + nr - 1) / nr : 0u;
        sCtl[10] = wr.z; sCtl[11] = wr.w;                    // first bin, first entry of the next bin (k_window_ranges)
    }
    __syncthreads();

    CLB_STAMP(1);
    // ------------------------------------------------------------------ phase A/B: reads -> counters
    const uint32_t t_low = (P.min_bq & 0x7fu) * 0x01010101u;
    uint2 *myDesc = sDesc + warp * 32;
    const uint32_t sLQ_s = smem_addr(sLQ);
    uint32_t acc_sum = 0;
    unsigned long long acc_mapq = 0;

    // Rounds of at most BPR batches of 32 reads: (A) walk the CIGARs, update the difference arrays and append the
    // M-segments to the CTA-wide pool; (B) after a barrier ALL warps stream the pooled segments slot by slot,
    // so the quality streaming is balanced across the CTA no matter how the batches fell.
    const uint32_t n_rounds = sCtl[8], bpr = sCtl[9];
    for (uint32_t round = 0; round < n_rounds; round++) {
    uint32_t *ctl = sCtl + 3 * (round & 1);
    const uint32_t rb1 = min(n_batches, (round + 1) * bpr);
    // (A) every lane owns up to two candidate reads per trip; the column loads of both are issued before anything
    //     depends on them, so a window pays two or three DRAM round trips in total instead of per batch.
    const uint32_t rr0 = r_lo + ((round * bpr) << 5), rr1 = min(r_hi, r_lo + (rb1 << 5));
    for (uint32_t i0 = rr0 + warp * 32; i0 < rr1; i0 += 2 * NT) {
        struct RMeta { int rel; uint32_t mq, c0, nops, lq, op0; uint64_t q0; };
        RMeta M[2];
        {
            uint32_t fl[2], c0[2], c1[2], mq[2], re[2]; int ps[2]; uint64_t q0[2], q1[2];
#pragma unroll
            for (int u = 0; u < 2; u++) {
                const uint32_t r = min(i0 + u * NT + lane, rr1 - 1);     // clamped lanes are discarded below
                fl[u] = P.flag[r]; c0[u] = P.cigar_off[r]; c1[u] = P.cigar_off[r + 1];
                ps[u] = P.pos[r]; mq[u] = P.mapq[r]; q0[u] = P.qual_off[r]; q1[u] = P.qual_off[r + 1];
                re[u] = P.read_end ? P.read_end[r] : 0xffffffffu;
            }
            uint32_t op0[2];
#pragma unroll
            for (int u = 0; u < 2; u++) op0[u] = c1[u] > c0[u] ? P.cigar[c0[u]] : 0xfu;
#pragma unroll
            for (int u = 0; u < 2; u++) {
                const bool live = (i0 + u * NT + lane < rr1) && !(fl[u] & 4u) && c1[u] > c0[u] && (long long)re[u] > W.wb;
                const uint64_t ql = q1[u] - q0[u];
                M[u].rel = (int)((long long)ps[u] - W.wb); M[u].mq = mq[u]; M[u].c0 = c0[u]; M[u].q0 = q0[u];
                M[u].lq = ql > 0xffffffffull ? 0xffffffffu : (uint32_t)ql;
                M[u].nops = live ? c1[u] - c0[u] : 0u; M[u].op0 = op0[u];
            }
        }
#pragma unroll 1                                                        // one copy of the walk: the executed code has to fit the instruction cache
        for (int u = 0; u < 2; u++) {
        if (i0 + u * NT >= rr1) break;                                   // warp-uniform
        const uint32_t bi = (i0 + u * NT - r_lo) >> 5;
        const uint32_t slab = W.lq_packed ? bi / BPA : 0u;
        const uint32_t lq_arr = sLQ_s + slab * (uint32_t)(LQ_SLAB * 4);
        const RMeta Mu = u ? M[1] : M[0];
        const int rel = Mu.rel; const uint32_t mq = Mu.mq, c0 = Mu.c0, nops = Mu.nops, lq = Mu.lq; const uint64_t q0 = Mu.q0;
        // short CIGARs are walked lane-serially (one loop trip per op, trip count = longest short CIGAR in the warp)
        bool cplx = nops > (uint32_t)FAST_OPS;
        if (__any_sync(FULL, !cplx && nops > 2u)) {                      // <= 2 ops cannot hold more than MAXSEG = 2 segments
            const uint32_t ncnt = cplx ? 0u : nops;
            const uint32_t kcnt = __reduce_max_sync(FULL, ncnt);
            uint32_t nm = 0;
            for (uint32_t k = 0; k < kcnt; k++) {
                const uint32_t op = k < ncnt ? (P.cigar[c0 + k] & 15u) : 15u;
                nm += (0x181u >> op) & 1u;                               // M, =, X
            }
            if (nm > (uint32_t)MAXSEG) cplx = true;                      // too many segments for the register slots
        }
        const uint32_t nfast = cplx ? 0u : nops;
        const uint32_t kmax = __reduce_max_sync(FULL, nfast);
        Seg sg0, sg1; bool h0 = false, h1 = false;
        {
            int rp = rel; uint32_t qp = 0;
            const bool pass = mq >= W.min_mapq;
            for (uint32_t k = 0; k < kmax; k++) {
                const uint32_t v = k < nfast ? (k == 0 ? Mu.op0 : P.cigar[c0 + k]) : 0xfu;  // op 15, len 0: no effect
                const uint32_t op = v & 15u, len = v >> 4;
                if (((0x181u >> op) & 1u) && pass) {
                    Seg s;
                    if (emit_m(W, lq_arr, rp, qp, len, q0, lq, s)) { if (!h0) { sg0 = s; h0 = true; } else { sg1 = s; h1 = true; } }
                }
                if (((0x18du >> op) & 1u) && rp < (int)WN) rp += (int)len;   // M, D, N, =, X consume the reference (saturates right of the window)
                if ((0x193u >> op) & 1u) qp += len;                          // M, I, S, =, X consume the query
            }
            if (nfast) emit_read<WIDE>(W, rel, rp, mq, acc_mapq);
        }
        {
            // pool append (warp-aggregated)
            const uint32_t nc0 = h0 ? seg_chunks(sg0) : 0u, nc1 = h1 ? seg_chunks(sg1) : 0u;
            const uint32_t bal0 = __ballot_sync(FULL, h0), bal1 = __ballot_sync(FULL, h1);
            const uint32_t n0 = __popc(bal0), n1 = __popc(bal1);
            if (n0 + n1) {
                const uint32_t mx = __reduce_max_sync(FULL, max(nc0, nc1));
                uint32_t base = 0;
                if (lane == 0) { base = atom_shared_add(smem_addr(&ctl[1]), n0 + n1); red_shared_max(smem_addr(&ctl[2]), mx); }
                base = __shfl_sync(FULL, base, 0);
                const uint32_t lt = (1u << lane) - 1u;
                if (h0) sPool[base + __popc(bal0 & lt)] = pack_desc(sg0, nc0, slab);
                if (h1) sPool[base + n0 + __popc(bal1 & lt)] = pack_desc(sg1, nc1, slab);
            }
        }

        // long CIGARs are queued for the whole CTA and expanded after the pool streaming, one read per warp at a time
        const uint32_t cmask = __ballot_sync(FULL, cplx);
        if (cmask) {
            uint32_t base = 0;
            if (lane == 0) base = atom_shared_add(smem_addr(&sCtl[16 + 2 * (round & 1)]), (uint32_t)__popc(cmask));
            base = __shfl_sync(FULL, base, 0);
            if (cplx) sCplx[(round & 1) * CPLX_CAP + base + __popc(cmask & ((1u << lane) - 1u))] = i0 + u * NT + lane;
        }
        }
    }
    __syncthreads();                                         // pool of this round is complete
    if (round == 0) CLB_STAMP(2);
    {
        const uint32_t pool_n = ctl[1], pool_s2 = (ctl[2] + 1u) >> 1;
        if (tid < 3) sCtl[3 * ((round + 1) & 1) + tid] = tid == 0 ? rb1 : 0u;     // next round's controls (nobody reads them before the barrier below)
        // the counter layout is a property of the window: one loop per layout keeps the test out of the per-chunk code
        if (W.lq_packed) process_slots<BQ_HI, 1>(W, sLQ_s, pool_n, pool_s2, sPool, sRcp, sMaskLo, sMaskHi, t_low, acc_sum, (uint32_t)tid, (uint32_t)NT);
        else process_slots<BQ_HI, 0>(W, sLQ_s, pool_n, pool_s2, sPool, sRcp, sMaskLo, sMaskHi, t_low, acc_sum, (uint32_t)tid, (uint32_t)NT);
        // queued long reads: warps pull one at a time (balanced no matter which groups they came from)
        const uint32_t ncp = sCtl[16 + 2 * (round & 1)];
        if (tid >= 2 && tid < 4) sCtl[16 + 2 * ((round + 1) & 1) + (tid - 2)] = 0u;
        for (;;) {
            uint32_t qi = 0;
            if (lane == 0) qi = atom_shared_add(smem_addr(&sCtl[17 + 2 * (round & 1)]), 1u);
            qi = __shfl_sync(FULL, qi, 0);
            if (qi >= ncp) break;
            const uint32_t r = sCplx[(round & 1) * CPLX_CAP + qi];
            const uint32_t c0 = P.cigar_off[r], c1 = P.cigar_off[r + 1];
            const uint64_t q0 = P.qual_off[r], ql = P.qual_off[r + 1] - q0;
            const uint32_t bi = (r - r_lo) >> 5;
            expand_long_read<BQ_HI, WIDE>(W, P, sLQ_s, W.lq_packed ? bi / BPA : 0u, (int)((long long)P.pos[r] - W.wb), P.mapq[r], c0, c1 - c0,
                                    ql > 0xffffffffull ? 0xffffffffu : (uint32_t)ql, q0, myDesc, sRcp, sMaskLo, sMaskHi, t_low, acc_sum,
                                    acc_mapq, lane);
        }
    }
    __syncthreads();                                         // counters final / pool free for the next round
    }
    if (n_rounds == 0) __syncthreads();
    CLB_STAMP(3);

    // ------------------------------------------------------------------ phase C: scan, classify, segment
    static_assert((size_t)DCAP * 8 >= 2 * DH_TAB * 4, "the depth table fits the segment pool");
    static_assert((size_t)DCAP * 8 >= 2 * DH_TAB * 4 + TL_SLOT_BYTES + NWARPS * 4, "the tile slots and run words fit the segment pool");
    static_assert((size_t)DCAP * 8 >= 2 * DH_TAB * 4 + TL_SLOT_BYTES + NWARPS * 4 + TH_SLOT_BYTES + TH_TAB * 4,
                  "the threshold slots and table fit the segment pool");
    static_assert((2 * DH_TAB * 4 + TL_SLOT_BYTES + NWARPS * 4) % 16 == 0, "threshold slots are 16-byte aligned");
    static_assert((size_t)DCAP * 8 >= 2 * DH_TAB * 4 + TL_SLOT_BYTES + NWARPS * 4 + TH_SLOT_BYTES + TH_TAB * 4 + NWARPS * 4,
                  "the QC run words fit the segment pool");
    uint32_t *sHist = reinterpret_cast<uint32_t *>(sPool);
    unsigned long long *sTileSum = reinterpret_cast<unsigned long long *>(sHist + 2 * DH_TAB);
    uint32_t *sTileFirst = reinterpret_cast<uint32_t *>(sTileSum + NWARPS * 8);
    uint32_t *sRunLast = sTileFirst + NWARPS;                              // per warp: its last raw depth (RUNS)
    uint32_t *sThSlot = sRunLast + NWARPS;                                 // THRESH: per-warp slots, then the nibble table
    uint32_t *sThTab = sThSlot + TH_SLOT_BYTES / 4;
    uint32_t *sQRunLast = sThTab + TH_TAB;                                 // per warp: its last QC depth (QRUNS)
    if constexpr (HIST) zero_depth_table(sHist);                           // the scan barrier below orders it before the counts
    if constexpr (THRESH) fill_thresh_table(sThTab, P);                    // ... and the table before count_tiles
    const uint32_t ebase = tid * PPT;
    uint32_t a[PPT], b[PPT], lqv[PPT], lw[WIDE ? PPT : 1];
    {
#pragma unroll
        for (int g = 0; g < PPT / 4; g++) {
            const uint4 av = *reinterpret_cast<const uint4 *>(sA + ebase + 4 * g), bv = *reinterpret_cast<const uint4 *>(sB + ebase + 4 * g);
            a[4 * g] = av.x; a[4 * g + 1] = av.y; a[4 * g + 2] = av.z; a[4 * g + 3] = av.w;
            b[4 * g] = bv.x; b[4 * g + 1] = bv.y; b[4 * g + 2] = bv.z; b[4 * g + 3] = bv.w;
        }
        if (WIDE) {
#pragma unroll
            for (int k = 0; k < PPT; k++) lw[WIDE ? k : 0] = sLowD[ebase + k];
        }
        if (W.lq_packed) {
            uint32_t ev[PPT / 4], od[PPT / 4];                  // 16-bit pair accumulators (4 entries per word)
#pragma unroll
            for (int g = 0; g < PPT / 4; g++) { ev[g] = 0; od[g] = 0; }
            for (uint32_t k = 0; k < n_lq; k++) {
                const uint32_t *row = sLQ + k * LQ_SLAB + 16 + (ebase >> 2);
#pragma unroll
                for (int g = 0; g < PPT / 4; g++) { const uint32_t q = row[g]; ev[g] += q & 0x00ff00ffu; od[g] += (q >> 8) & 0x00ff00ffu; }
            }
#pragma unroll
            for (int g = 0; g < PPT / 4; g++) {
                lqv[4 * g] = ev[g] & 0xffffu; lqv[4 * g + 1] = od[g] & 0xffffu; lqv[4 * g + 2] = ev[g] >> 16; lqv[4 * g + 3] = od[g] >> 16;
            }
        } else {
#pragma unroll
            for (int g = 0; g < PPT / 4; g++) {
                const uint4 qv = *reinterpret_cast<const uint4 *>(sLQ + 16 + ebase + 4 * g);
                lqv[4 * g] = qv.x; lqv[4 * g + 1] = qv.y; lqv[4 * g + 2] = qv.z; lqv[4 * g + 3] = qv.w;
            }
        }
    }
#pragma unroll
    for (int k = 1; k < PPT; k++) { a[k] += a[k - 1]; b[k] += b[k - 1]; if (WIDE) lw[WIDE ? k : 0] += lw[WIDE ? k - 1 : 0]; }
    {
        const uint32_t ta = a[PPT - 1], tb = b[PPT - 1], tl = WIDE ? lw[WIDE ? PPT - 1 : 0] : 0u;
        uint32_t ia = ta, ib = tb, il = tl;
#pragma unroll
        for (int dd = 1; dd < 32; dd <<= 1) {
            const uint32_t t1 = __shfl_up_sync(FULL, ia, dd), t2 = __shfl_up_sync(FULL, ib, dd);
            if (lane >= dd) { ia += t1; ib += t2; }
            if (WIDE) { const uint32_t t3 = __shfl_up_sync(FULL, il, dd); if (lane >= dd) il += t3; }
        }
        if (lane == 31) { sScan[warp] = ia; sScan[NWARPS + warp] = ib; if (WIDE) sScan[4 * NWARPS + warp] = il; }
        __syncthreads();
        // totals of the warps before this one: lane j holds warp j's total, one REDUX per array sums lanes < warp
        const bool before = lane < warp;
        uint32_t oa = ia - ta + __reduce_add_sync(FULL, before ? sScan[lane] : 0u);
        uint32_t ob = ib - tb + __reduce_add_sync(FULL, before ? sScan[NWARPS + lane] : 0u);
        uint32_t ol = il - tl;
        if (WIDE) ol += __reduce_add_sync(FULL, before ? sScan[4 * NWARPS + lane] : 0u);
#pragma unroll
        for (int k = 0; k < PPT; k++) { a[k] += oa; b[k] += ob; if (WIDE) lw[WIDE ? k : 0] += ol; }
    }
    // REF_N bits of this thread's entries
    uint32_t nbits;
    {
        const long long p0 = W.wb + (long long)ebase;
        if (p0 >= 0) { const uint32_t wi = (uint32_t)(p0 >> 5); nbits = __funnelshift_r(P.nmask[wi], P.nmask[wi + 1], (uint32_t)(p0 & 31)); }
        else nbits = P.nmask[0] << 1;
    }
    using Sum = typename std::conditional<WIDE, unsigned long long, uint32_t>::type;   // deep windows: 32-bit partial sums could overflow
    Entries<Sum> e = entries_of<Sum>(ebase, ebase == 0 ? 1u : 0u, n_ent);              // entry 0 is the halo
    const StateLimits lim = state_limits(P);
    DepthHist dh{};
    if constexpr (HIST) dh = depth_hist_of(smem_addr(sHist), P);
    // Two copies of the per-entry classification, chosen per thread: when none of the thread's entries is deeper than
    // the shared-memory threshold table the lookup is a plain LDS; otherwise every entry may go to the global table
    // (kept apart because those loads, predicated off, would still cost six issue slots per ordinary entry).
    auto classify = [&](auto deep_tag) {
        constexpr bool DEEP = decltype(deep_tag)::value;
#pragma unroll
        for (int k = 0; k < PPT; k++) {
            const uint32_t raw = WIDE ? a[k] : a[k] & 0xffffu, low = WIDE ? lw[WIDE ? k : 0] : a[k] >> 16;
            const uint32_t qc = b[k] - lqv[k];
            uint32_t fst;
            if (DEEP) {
                fst = sFirst[min(raw, (uint32_t)NFIRST - 1u)];
                if (raw >= (uint32_t)NFIRST) fst = (WIDE && raw >= 65536u) ? first_low(raw, P.max_low_mapq_fraction) : P.first_tab[raw];
            } else {
                fst = sFirst[raw];
            }
            classify_entry(e, k, raw, low, qc, fst, (nbits >> k) & 1u, lim);
            if constexpr (HIST) count_depth<false>(dh, e, k, raw, qc);
            b[k] = qc;                                                    // keep qc (entry 0 below, optional debug dump)
        }
    };
    {
        uint32_t deepest = 0;                                             // an upper bound of the thread's raw depths
#pragma unroll
        for (int k = 0; k < PPT; k++) deepest |= WIDE ? a[k] : a[k] & 0xffffu;
        if (deepest < (uint32_t)NFIRST) classify(std::false_type{}); else classify(std::true_type{});
    }
    if constexpr (HIST) close_depth_runs<false>(dh);
    if (!(e.vmask & 1u)) {
        // the halo entry (thread 0) is a real position and carries depth: take it out of the sums again (reads are clipped
        // at the region end, so entries past it have none)
        const uint32_t raw0 = WIDE ? a[0] : a[0] & 0xffffu;
        e.covered -= raw0 > 0 ? 1u : 0u; e.sraw -= raw0; e.sqc -= b[0];
    }
    close_entries(e, n_ent, sLast, sScan);
    const auto raw_of = [&](int k) { return WIDE ? a[k] : a[k] & 0xffffu; };   // not the packed word: its high half is the low-MAPQ depth
    const auto qc_of = [&](int k) { return b[k]; };                        // the QC depth since the classify loop, halo included
    if constexpr (RUNS) publish_run_depth(e, n_ent, raw_of, sRunLast, sScan + 3 * NWARPS + 2);
    if constexpr (QRUNS) publish_run_depth(e, n_ent, qc_of, sQRunLast, sScan + 3 * NWARPS + 4);
    dbg_dump<DBG>(e, (uint32_t)(W.wb - P.region_start),
                  [&](int k) { return make_uint3(WIDE ? a[k] : a[k] & 0xffffu, b[k], WIDE ? lw[WIDE ? k : 0] : a[k] >> 16); }, P);
    if constexpr (TILES)
        count_tiles<THRESH>(e, (uint32_t)W.wb, nbits, [&](int k) { return make_uint2(WIDE ? a[k] : a[k] & 0xffffu, b[k]); }, sTileSum,
                            sTileFirst, P, sThTab, sThSlot);
    reduce_stats(e, acc_sum, acc_mapq, sWStats, P);
    if constexpr (HIST) flush_depth_table(dh, sHist);                      // after reduce_stats' barrier
    if constexpr (TILES) flush_tiles<THRESH>(sTileSum, sTileFirst, P, sThSlot);
    CLB_STAMP(4);
    // entry 1 of window 0 is the region's first position: it always starts a record, soft when it merely continues the
    // previous shard's run; it always starts a raw and a QC depth run too (the halo is compared with for every other window)
    const uint32_t region_first = w == 0 && tid == 0 ? 2u : 0u;
    const uint32_t rmask = RUNS ? run_starts(e, raw_of, region_first, sRunLast) : 0u;
    const uint32_t qmask = QRUNS ? run_starts(e, qc_of, region_first, sQRunLast) : 0u;
    write_records<RUNS, QRUNS>(e, (uint32_t)W.wb, region_first, P.region_start != 0 ? region_first : 0u, 0u, sLast, sScan, w, P, rmask,
                               raw_of, qmask, qc_of);
    CLB_STAMP(5);
    add_bins(e, (uint32_t)W.wb, 1u, n_ent, sCtl[10], sCtl[11], P);        // first bin, next bin's entry: divided out once by thread 0
    CLB_STAMP(6);
    CLB_STAMP_VALUE(7, r_hi - r_lo);
}

// General kernel: persistent CTAs take the windows queued by k_window_ranges / k_pileup_fast one ticket at a time.
// The queue only grows between launches (all pushes of a batch of windows happen before this kernel starts on the
// same stream), so a CTA that draws a ticket past the end gives it back and leaves: gen_taken == gen_count afterwards.
template <bool BQ_HI, bool DBG, unsigned FEAT = 0u>
__global__ void __launch_bounds__(NT, CLB_MINB) k_pileup_general(const KParams P) {
    __shared__ uint32_t s_ticket;
    const uint32_t n = *P.gen_count;
    const bool refused = (*P.err & ERR_INPUT_REFUSED) != 0;             // take the tickets, do not walk the columns
    for (;;) {
        if (threadIdx.x == 0) {
            uint32_t t = atomicAdd(P.gen_taken, 1u);
            if (t >= n) { atomicSub(P.gen_taken, 1u); t = 0xffffffffu; }
            s_ticket = t;
        }
        __syncthreads();
        const uint32_t t = s_ticket;
        if (t == 0xffffffffu) break;
        if (!refused) pileup_classify_window<BQ_HI, false, DBG, FEAT>(P, P.gen_list[t]);
        __syncthreads();                                     // shared memory (and s_ticket) are reused by the next window
    }
}

// Second pass over the (rare) windows k_pileup_classify queued because they hold more than 65535 candidate reads:
// a fixed small grid walks the queue; with an empty queue the launch costs a few microseconds.
template <bool BQ_HI, bool DBG, unsigned FEAT = 0u>
__global__ void __launch_bounds__(NT, 1) k_pileup_classify_deep(const KParams P) {
    if (*P.err & ERR_RESULT_INVALID) return;
    const uint32_t n = *P.deep_count;
    for (uint32_t i = blockIdx.x; i < n; i += gridDim.x) {
        pileup_classify_window<BQ_HI, true, DBG, FEAT>(P, P.deep_list[i]);
        __syncthreads();                                     // shared memory is reused by the next window
    }
}

// ---------------------------------------------------------------------------------------------
// Small helper kernels
// ---------------------------------------------------------------------------------------------
#ifndef CLB_WR_LANES
#define CLB_WR_LANES 8
#endif
constexpr int WR_LANES = CLB_WR_LANES;   // lanes that share one window in k_window_ranges (a power of two <= 32)
static_assert(WR_LANES >= 2 && WR_LANES <= 32 && (WR_LANES & (WR_LANES - 1)) == 0, "lane group");

// Lower bound by a group of GS lanes: GS probes per round trip (the range shrinks (GS + 1)-fold per step).  gmask = the
// group's lanes, gl = lane within the group, gbase = first lane of the group.
__device__ __forceinline__ uint32_t lower_bound_pos_group(const int32_t *pos, uint32_t n, long long key, uint32_t gmask, int gl, int gbase) {
    constexpr uint32_t GS = WR_LANES;
    uint32_t lo = 0, hi = n;                             // the answer lies in [lo, hi]
    while (hi - lo > GS) {
        const uint32_t idx = lo + (uint32_t)(((unsigned long long)(hi - lo) * (unsigned)(gl + 1)) / (GS + 1u));   // lo < idx < hi, increasing with the lane
        const uint32_t below = (__ballot_sync(gmask, (long long)pos[idx] < key) >> gbase) & (GS == 32u ? 0xffffffffu : ((1u << GS) - 1u));   // a run of ones, then zeros
        const int c = __popc(below);
        const uint32_t lo_n = __shfl_sync(gmask, idx, gbase + max(c - 1, 0)) + 1u;
        const uint32_t hi_n = __shfl_sync(gmask, idx, gbase + min(c, (int)GS - 1));
        lo = c ? lo_n : lo; hi = c < (int)GS ? hi_n : hi;
    }
    const uint32_t i = lo + (uint32_t)gl;
    return lo + (uint32_t)__popc(__ballot_sync(gmask, i < hi && (long long)pos[i] < key) & gmask);
}

// candidate read range of every window: reads with pos < window end and pos + max_span > halo position; and the
// window's class: shard-first windows (they need the state of the base before the shard), windows of long-read contigs
// and windows whose candidate count or CIGAR density cannot be an ordinary short-read pile go straight to the general queue.
// A group of WR_LANES lanes per window: the searches probe WR_LANES positions per step and the two verification loops are
// spread over the group.  The kernel is bound by (dependent round trips per window) x (waves of warps): one thread per
// window spent 82 us of a chr1 step in ~70 round trips, a whole warp per window 12 round trips but 13 waves of warps.
__global__ void k_window_ranges(const int32_t *pos, uint32_t n_reads, uint32_t region_start, uint32_t region_end,
                                const uint32_t *max_span_ptr, uint32_t w_first, uint32_t n_w,
                                const uint64_t *qual_off, const uint32_t *cigar_off, uint32_t stride, uint4 *win_rec,
                                uint32_t force_general, uint32_t *gen_list, uint32_t *gen_count, const uint32_t *max_qlen_ptr) {
    constexpr uint32_t GS = WR_LANES;
    const uint32_t gi = (blockIdx.x * blockDim.x + threadIdx.x) / GS;     // window of this group (groups past the end run a clamped copy: whole warps stay converged)
    const int lane = threadIdx.x & 31, gl = lane & (int)(GS - 1u), gbase = lane - gl;
    const uint32_t gmask = (GS == 32u ? 0xffffffffu : ((1u << GS) - 1u)) << gbase;
    const bool real = gi < n_w;
    const uint32_t i = real ? gi : n_w - 1u;
    const uint32_t max_span = *max_span_ptr;
    const uint32_t w = w_first + i;
    const long long wb = (long long)region_start + (long long)w * WREAL - 1;
    const long long wend = min(wb + WN, (long long)region_end);
    const uint32_t r_lo = lower_bound_pos_group(pos, n_reads, wb - (long long)max_span + 1, gmask, gl, gbase);
    const uint32_t r_hi = lower_bound_pos_group(pos, n_reads, wend, gmask, gl, gbase);
    const uint32_t first_bin = stride ? (uint32_t)(wb + 1) / stride : 0u;
    const uint64_t q_lo = qual_off[r_lo] & ~15ull, q_hi = qual_off[r_hi];
    const uint32_t n_cand = r_hi - r_lo;
    bool general = force_general != 0 || (w == 0 && region_start != 0) || n_cand > 16384u || q_hi - q_lo > 0xfffffff0ull;
    const uint32_t c_lo = cigar_off[r_lo], c_hi = cigar_off[r_hi];
    if (!general && n_cand) general = (c_hi - c_lo) > 8u * n_cand + 64u;
    // the fast kernel's depth proof (pos[i] - pos[i - 254] >= max_span for every candidate), sampled: a deep pile fails it
    // at the first sample and goes to the general kernel without a wasted attempt
    if (!general) {
        bool deep = false;
        for (uint32_t i2 = r_lo + 254u * (uint32_t)(gl + 1); i2 < r_hi; i2 += 254u * GS)
            deep |= (long long)pos[i2 - 254u] + (long long)max_span > (long long)pos[i2];
        general = (__ballot_sync(gmask, deep) & gmask) != 0u;
    }
    // Sub-batches of the fast kernel: G <= 32 reads at a time (one per lane) whose qualities fit a warp's stage.  Start
    // from the mean read length of the window and verify every sub-batch; shrink a few times before giving up.
    uint32_t G = 32;
    if (!general && n_cand) {
        const uint64_t total = q_hi - q_lo;
        if (total * 32u > (uint64_t)(CLB_F_WSTAGE - 16) * n_cand) G = (uint32_t)(((uint64_t)(CLB_F_WSTAGE - 16) * n_cand) / total);
        // no sub-batch of G reads can outgrow the stage when even G reads of the contig's longest quality string fit (k_validate_batch
        // tracks that maximum): uniform-length reads skip the verification, which touches qual_off once per sub-batch
        const uint32_t max_qlen = *max_qlen_ptr;
        bool ok = G >= 4u && max_qlen != 0u && (uint64_t)G * max_qlen + 32u <= (uint64_t)CLB_F_WSTAGE;
        for (int tries = 0; tries < 4 && G >= 4u && !ok; tries++) {
            uint32_t worst = 0;                          // staged bytes of the largest sub-batch, saturated
            for (uint32_t b = r_lo + (uint32_t)gl * G; b < r_hi; b += GS * G) {
                const uint64_t bytes = (qual_off[min(b + G, r_hi)] - (qual_off[b] & ~15ull) + 15ull) & ~15ull;
                worst = max(worst, (uint32_t)min(bytes, (uint64_t)0xffffffffu));
            }
            ok = __reduce_max_sync(gmask, worst) <= (uint32_t)CLB_F_WSTAGE;
            if (!ok) G -= max(1u, G / 8u);
        }
        if (!ok) general = true;
    }
    if (real && gl == 0) {
        win_rec[3 * (size_t)w] = make_uint4(r_lo, r_hi, first_bin, stride ? (uint32_t)((long long)(first_bin + 1) * stride - wb) : 0xffffffffu);
        *reinterpret_cast<ulonglong2 *>(win_rec + 3 * (size_t)w + 1) = make_ulonglong2(q_lo, q_hi);
        win_rec[3 * (size_t)w + 2] = make_uint4(general ? 0u : G, general ? 0u : (n_cand + G - 1u) / G, c_lo, c_hi);   // reads per sub-batch, sub-batches, CIGAR op range
        if (general) gen_list[atomicAdd(gen_count, 1u)] = w;
    }
}

// pos + reference span of every read, and the maximum span (long-read mode / max_ref_span == 0)
__global__ void k_read_end(const int32_t *pos, const uint32_t *cigar_off, const uint32_t *cigar, uint32_t r0, uint32_t r1,
                           uint32_t *read_end, uint32_t *max_span) {
    const uint32_t r = r0 + blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t span = 0;
    if (r < r1) {
        for (uint32_t c = cigar_off[r]; c < cigar_off[r + 1]; c++) { const uint32_t v = cigar[c]; if (op_ref(v & 15u)) span += v >> 4; }
        if (read_end) read_end[r] = (uint32_t)pos[r] + span;
    }
    span = __reduce_max_sync(FULL, span);
    if (max_span && (threadIdx.x & 31) == 0 && span) atomicMax(max_span, span);
}

// Long-read mode: one warp per read walks the CIGAR once, 32 ops per step aligned to the contig-wide CIGAR column, and
// records the read's cumulative (reference, query) offsets at every 32-op boundary inside it, its end and the maximum span.
__global__ void k_cigar_checkpoints(const int32_t *pos, const uint32_t *cigar_off, const uint32_t *cigar, uint32_t r0, uint32_t r1,
                                    uint32_t *read_end, uint32_t *max_span, uint2 *ckpt) {
    const uint32_t r = r0 + ((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (r >= r1) return;
    const uint32_t c0 = cigar_off[r], c1 = cigar_off[r + 1];
    uint32_t ob = c0, cr = 0, cq = 0;
    while (ob < c1) {
        const uint32_t bend = min(c1, (ob | 31u) + 1u);
        const uint32_t v = (ob + lane < bend) ? cigar[ob + lane] : 0xfu;
        const uint32_t op = v & 15u, len = v >> 4;
        cr += __reduce_add_sync(FULL, ((0x18du >> op) & 1u) ? len : 0u);
        cq += __reduce_add_sync(FULL, ((0x193u >> op) & 1u) ? len : 0u);
        ob = bend;
        if (ob < c1 && lane == 0) ckpt[ob >> 5] = make_uint2(cr, cq);
    }
    if (lane == 0) { if (read_end) read_end[r] = (uint32_t)pos[r] + cr; if (max_span && cr) atomicMax(max_span, cr); }
}

// batch append, step 1: validate ordering of the freshly copied (still batch-relative) columns.
// Device entries r0+1 .. r0+n hold the batch's offsets[1..n]; entry r0 is the previous batch's end.
__global__ void k_validate_batch(const int32_t *pos, const uint32_t *cigar_off, const uint64_t *qual_off, uint32_t r0, uint32_t n,
                                 uint32_t *err, uint32_t *max_qlen) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t ql = 0;
    if (i < n) {
        if (pos[r0 + i] < 0 || (r0 + i > 0 && pos[r0 + i] < pos[r0 + i - 1])) atomicOr(err, ERR_UNSORTED);
        const uint32_t cprev = i == 0 ? 0u : cigar_off[r0 + i];
        const uint64_t qprev = i == 0 ? 0ull : qual_off[r0 + i];
        const uint64_t qnext = qual_off[r0 + i + 1];
        if (cigar_off[r0 + i + 1] < cprev || qnext < qprev) atomicOr(err, ERR_OFFSETS);
        ql = qnext >= qprev ? (uint32_t)min(qnext - qprev, (uint64_t)0xffffffffu) : 0xffffffffu;
    }
    // longest quality string of the contig (saturated): k_window_ranges sizes the fast kernel's sub-batches with it
    const uint32_t wmax = __reduce_max_sync(FULL, ql);               // every lane of the warp is here
    if ((threadIdx.x & 31) == 0 && wmax) atomicMax(max_qlen, wmax);
}
// step 2: rebase entries r0+1 .. r0+n onto the contig-wide payload arrays
__global__ void k_rebase_batch(uint32_t *cigar_off, uint64_t *qual_off, uint32_t r0, uint32_t n, uint32_t cigar_base, uint64_t qual_base) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    cigar_off[r0 + i + 1] += cigar_base;
    qual_off[r0 + i + 1] += qual_base;
}

// ASCII reference -> bit-packed N mask, one 32-bit word (32 bases, two 16-byte loads) per thread; bases past ref_len (but
// inside the contig) read as 'N' (mod.rs:79-80).  ref is 256-byte aligned (cudaMalloc) and padded to a multiple of 32 bytes.
__global__ void k_nmask_from_ascii(const uint8_t *ref, uint64_t ref_len, uint32_t contig_len, uint32_t *nmask, uint32_t n_words) {
    const uint64_t wi = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (wi >= n_words) return;
    const uint64_t p0 = wi * 32ull;
    uint32_t word = 0;
    if (p0 + 32ull <= ref_len) {
        const uint4 a = reinterpret_cast<const uint4 *>(ref + p0)[0], b = reinterpret_cast<const uint4 *>(ref + p0)[1];
        const uint32_t v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const uint32_t x = (v[k] | 0x20202020u) ^ 0x6e6e6e6eu;          // zero byte <=> 'N' or 'n'
            const uint32_t z = ~(((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & 0x80808080u;   // 0x80 in every zero byte
            word |= (((z >> 7) & 1u) | ((z >> 14) & 2u) | ((z >> 21) & 4u) | ((z >> 28) & 8u)) << (4 * k);
        }
    } else {
        for (uint32_t j = 0; j < 32; j++) {
            const uint64_t p = p0 + j;
            bool isn = false;
            if (p < ref_len) { const uint8_t c = ref[p]; isn = (c == 'N' || c == 'n'); }
            else if (p < contig_len) isn = true;
            word |= (isn ? 1u : 0u) << j;
        }
    }
    nmask[wi] = word;
}

// first_tab[raw] = smallest low in [0, raw+1] with (double)low / (double)raw > fraction  (callable_profiler.rs:100-101)
// The small tables every window keeps in shared memory, laid out as the kernel expects them:
//   17 x uint4 "bytes below lo" masks | 17 x uint4 "bytes at/above hi" masks | first_tab[0..NFIRST) | ceil(2^32 / i) for i < NRCP
__global__ void k_window_tables(uint32_t *out, double fraction) {
    const uint32_t t = threadIdx.x;
    if (t < 17) {
#pragma unroll
        for (int q = 0; q < 4; q++) {
            uint32_t ml = 0, mh = 0;
#pragma unroll
            for (int j = 0; j < 4; j++) {
                if (4 * q + j < (int)t) ml |= 0xffu << (8 * j);          // bytes below lo = t
                if (4 * q + j >= (int)t) mh |= 0xffu << (8 * j);         // bytes at/above hi = t
            }
            out[4 * t + q] = ml; out[17 * 4 + 4 * t + q] = mh;
        }
    }
    for (uint32_t i = t; i < (uint32_t)NFIRST; i += blockDim.x) out[2 * 17 * 4 + i] = first_low(i, fraction);
    for (uint32_t i = t; i < (uint32_t)NRCP; i += blockDim.x) out[2 * 17 * 4 + NFIRST + i] = i > 1 ? 0xffffffffu / i + 1u : 0u;
}

__global__ void k_first_table(uint32_t *first_tab, uint8_t *first_tab8, double fraction) {
    const uint32_t raw = blockIdx.x * blockDim.x + threadIdx.x;
    if (raw >= 65536u) return;
    const uint32_t f = first_low(raw, fraction);
    first_tab[raw] = f;
    if (raw < 256u) first_tab8[raw] = (uint8_t)min(f, 255u);       // f <= raw + 1; depth 0 is NO_COVERAGE whatever the table says
}

// ---------------------------------------------------------------------------------------------
// Interval compaction: per-window record chunks (arbitrary order) -> sorted clb_interval array
// ---------------------------------------------------------------------------------------------
// The same three steps compact the depth runs, raw and QC (Tab = uint4: KParams::run_win_tab / qrun_win_tab, records uint2,
// copied as they are).
// step 1: every block scans 1024 windows locally and publishes its total
template <typename Tab>
__global__ void __launch_bounds__(1024) k_scan_windows_local(const Tab *win_tab, uint32_t n_w, uint32_t *win_out, uint32_t *blk_tot,
                                                             const uint32_t *err) {
    __shared__ uint32_t sW[32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (*err & ERR_RESULT_INVALID) return;                    // win_tab was not written: nothing to scan
    const uint32_t i = blockIdx.x * 1024u + tid;
    const uint32_t v = i < n_w ? win_count(win_tab[i]) - win_drop_first(win_tab, i) : 0u;
    uint32_t inc = v;
#pragma unroll
    for (int dd = 1; dd < 32; dd <<= 1) { const uint32_t t = __shfl_up_sync(FULL, inc, dd); if (lane >= dd) inc += t; }
    if (lane == 31) sW[warp] = inc;
    __syncthreads();
    const uint32_t wt = sW[lane];
    const uint32_t off = __reduce_add_sync(FULL, lane < warp ? wt : 0u);
    if (i < n_w) win_out[i] = off + inc - v;
    if (tid == 1023) blk_tot[blockIdx.x] = off + inc;
}
// step 2: one block turns the block totals into block offsets (in place) and the grand total
__global__ void __launch_bounds__(1024) k_scan_blocks(uint32_t *blk_tot, uint32_t n_blk, uint32_t *n_total) {
    __shared__ uint32_t sW[32];
    __shared__ uint32_t sCarry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) sCarry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n_blk; base += 1024u) {
        const uint32_t i = base + tid;
        const uint32_t v = i < n_blk ? blk_tot[i] : 0u;
        uint32_t inc = v;
#pragma unroll
        for (int dd = 1; dd < 32; dd <<= 1) { const uint32_t t = __shfl_up_sync(FULL, inc, dd); if (lane >= dd) inc += t; }
        if (lane == 31) sW[warp] = inc;
        __syncthreads();
        const uint32_t wt = sW[lane];
        const uint32_t off = sCarry + __reduce_add_sync(FULL, lane < warp ? wt : 0u);
        if (i < n_blk) blk_tot[i] = off + inc - v;
        __syncthreads();
        if (tid == 1023) sCarry = off + inc;
        __syncthreads();
    }
    if (tid == 0) *n_total = sCarry;
}

// one warp per window: move its records to their sorted place (start/state/soft; end filled next)
// (nothing to gather when the record buffer overflowed: the records past its capacity were never written and the
// interval array is just as small; the host grows both and re-runs the contig.  Nothing either when the input was refused:
// win_tab and the scan hold whatever an earlier contig, or no contig, left there)
// (the depth runs of a contig whose state records overflowed are not gathered either: the host re-runs it)
template <typename Tab, typename Rec, typename Out>
__global__ void k_gather_intervals(const Rec *rec, const Tab *win_tab, const uint32_t *win_out, const uint32_t *blk_off,
                                   uint32_t n_w, Out *out, const uint32_t *err) {
    const uint32_t w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (w >= n_w || (*err & (ERR_REC_OVERFLOW | ERR_RESULT_INVALID))) return;
    const Tab t = win_tab[w];
    const uint32_t skip = win_drop_first(win_tab, w);
    const uint32_t o = blk_off[w >> 10] + win_out[w], cnt = win_count(t) - skip;
    for (uint32_t i = lane; i < cnt; i += 32) {
        out[o + i] = gather_out(rec[t.x + skip + i]);
    }
}

__global__ void k_fill_ends(IntervalOut *out, const uint32_t *n_total, uint32_t region_end, const uint32_t *err) {
    if (*err & (ERR_REC_OVERFLOW | ERR_RESULT_INVALID)) return;
    const uint32_t n = *n_total;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        out[i].end = (i + 1 < n) ? out[i + 1].start : region_end;
}

// padded per-counter lines -> compact [N_STATS] prefix of the counter buffer (bins follow it)
__global__ void k_pack_stats(const unsigned long long *stats_padded, unsigned long long *counters) {
    if (threadIdx.x < N_STATS) counters[threadIdx.x] = stats_padded[threadIdx.x * STAT_STRIDE];
}

// the DH_SLOTS copies of the depth histograms ([raw n][qc n] each, n2 = 2n words) -> their place in the counter buffer
__global__ void k_fold_depth_hist(const unsigned long long *slots, uint32_t n2, unsigned long long *out) {
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += gridDim.x * blockDim.x) {
        unsigned long long t = 0;
#pragma unroll
        for (int k = 0; k < DH_SLOTS; k++) t += slots[(size_t)k * n2 + i];
        out[i] = t;
    }
}

}  // namespace clb
