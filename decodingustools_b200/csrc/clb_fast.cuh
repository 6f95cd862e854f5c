// clb_fast.cuh -- the fast window kernel of the CallableLoci hot path (sm_100a).
//
// Same reference loop as clb_kernels.cuh (mod.rs:17-42,65-120, callable_profiler.rs:89-155, contig_profiler.rs:47-83,
// histogram_plotter.rs:74-102), restructured for the ordinary window: short CIGARs and fewer than 255 reads over any
// position.  Anything else (long reads, deep piles, a shard's first window) is queued for k_pileup_general, the
// round-1 kernel, so results never depend on which kernel took a window.
//
// What is different from the general kernel, and why (ncu of round 1: issue bound at 0.416 warp instructions per cell):
//   * Every warp runs its own pipeline over sub-batches of <= 32 consecutive reads (one per lane).  The qualities of a
//     sub-batch are ONE contiguous byte range: lane 0 moves it into the warp's stage with a single cp.async.bulk (TMA
//     engine, completion on the warp's own mbarrier) and the CIGAR walk of the 32 reads runs while the copy is in
//     flight.  No per-thread address math for the qualities, no LDG wavefronts, no descriptor pool, no CTA barrier
//     until phase C.
//   * Every thread then streams ITS OWN read's M-segment from shared memory with LDS.128: the segment lives in
//     registers, interior chunks need no byte masks, the loop is 6 instructions per 4 bases.
//   * Base-quality PASS counts go to four packed-u8 arrays selected by (entry of chunk byte 0) mod 4, so the four
//     words of a chunk are added with four plain shared atomics and no funnel shifts; qc depth is the sum of the
//     four arrays (phase C realigns them once per 8 entries), which also removes the M-coverage difference array.
//     A byte cannot overflow because the window is only taken when pos[i] - pos[i - 254] >= max_ref_span for every
//     candidate read, i.e. fewer than 255 reads cover any position.
//   * No halo entry: a window always emits a record for its first position, flagged "window soft", and the
//     interval gather drops it when the previous window ended in the same state.
#pragma once
#include "clb_kernels.cuh"

namespace clb {

constexpr int F_CW = 520;                 // words per alignment-class array (2048 / 4 + 8; 520 % 32 == 8 staggers the banks)
constexpr int F_WSTAGE = CLB_F_WSTAGE;    // staged quality bytes per warp and sub-batch of <= 32 reads (k_window_ranges sizes the sub-batches)
constexpr int F_XCAP = 96;                // second-and-later M-segments per window (streamed from global memory at the end; more: general kernel)
constexpr int F_MAXOPS = 64;              // longest CIGAR walked lane-serially
constexpr int F_LOOKBACK = 254;           // depth proof: pos[i] - pos[i - 254] >= max span  =>  depth <= 254 everywhere
constexpr int F_NFIRST = 256;             // low-MAPQ threshold table entries, one byte each (raw depth <= 254)
#ifndef CLB_F_MINB
#define CLB_F_MINB 4
#endif

// shared memory: A | C (4 class arrays) | one stage per warp | X list | byte masks | first table (u8) | control words | one mbarrier per warp.
// The scratch of phase C (scan, last states, warp stats) reuses the stages, which are idle by then.
constexpr int F_OFF_A = 0;
constexpr int F_OFF_C = F_OFF_A + WN * 4;
constexpr int F_OFF_STAGE = F_OFF_C + 4 * F_CW * 4;
constexpr int F_OFF_X = F_OFF_STAGE + NWARPS * F_WSTAGE;
constexpr int F_OFF_MASK = F_OFF_X + F_XCAP * 8;
constexpr int F_OFF_FIRST = F_OFF_MASK + 2 * 17 * 16;
constexpr int F_OFF_CTL = F_OFF_FIRST + F_NFIRST;
constexpr int F_OFF_BAR = F_OFF_CTL + 16 * 4;
constexpr size_t F_SMEM = F_OFF_BAR + NWARPS * 8;
constexpr int F_OFF_SCAN = F_OFF_STAGE;                        // phase C scratch inside the stages
constexpr int F_OFF_LAST = F_OFF_SCAN + 64 * 4;
constexpr int F_OFF_WSTATS = F_OFF_LAST + NT;
constexpr int F_OFF_HIST = F_OFF_WSTATS + NWARPS * N_STATS * 8;    // depth table (HIST instantiations), 2 x DH_TAB u32
constexpr int F_OFF_TILE = F_OFF_HIST + 2 * DH_TAB * 4;              // tile slots (TILES instantiations), TL_SLOT_BYTES
constexpr int F_OFF_RUN = F_OFF_TILE + TL_SLOT_BYTES;                 // per warp its last raw depth (RUNS instantiations), u32
static_assert(F_OFF_STAGE % 16 == 0 && F_WSTAGE % 16 == 0, "bulk copies need 16-byte aligned destinations");
static_assert(F_OFF_WSTATS % 8 == 0 && F_OFF_BAR % 8 == 0 && F_OFF_X % 8 == 0 && F_OFF_MASK % 16 == 0 && F_OFF_FIRST % 16 == 0, "alignment");
static_assert(F_OFF_RUN + NWARPS * 4 <= F_OFF_X, "phase C scratch fits the stages");
static_assert(CLB_F_MINB * (F_SMEM + 1024) <= 228 * 1024, "shared memory per SM");
enum { FC_BAIL = 0, FC_XCNT = 1 };

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" :: "r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" :: "r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    } while (!done);
}
// global -> shared bulk copy (TMA engine), completion counted in bytes on the mbarrier
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t saddr) {
    uint4 r = make_uint4(0, 0, 0, 0);
    if (!CLB_SMEM_OK(saddr, 16u)) return r;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(saddr));
    return r;
}

// 0x80 in every byte of x that is >= T (unsigned).  t_low = (T & 0x7f) * 0x01010101; BQ_HI = (T >= 128).
template <bool BQ_HI>
__device__ __forceinline__ uint32_t bytes_ge(uint32_t x, uint32_t t_low) {
    const uint32_t H = 0x80808080u;
    const uint32_t d = (x | H) - t_low;                  // bit7 = ((x & 0x7f) >= (T & 0x7f)), no cross-byte borrow
    return (BQ_HI ? (x & d) : (x | d)) & H;
}

__device__ __forceinline__ uint4 or4(const uint4 a, const uint4 b) { return make_uint4(a.x | b.x, a.y | b.y, a.z | b.z, a.w | b.w); }

// One 16-byte chunk: pass flags of the bytes not in drop (0xFF in bytes outside the segment), acc += 128 x the sum of the
// passing qualities (the 0x80 flags are the dot-product weights), the four flag words added to dst .. dst + 12.  An interior
// chunk passes a zero drop mask: 6 instructions per word (LOP3, IMAD, LOP3, SHF, IDP.4A, ATOMS).
template <bool BQ_HI>
__device__ __forceinline__ void count_words(const uint4 v, const uint4 drop, uint32_t dst, uint32_t t_low, uint32_t &acc) {
    const uint32_t l0 = bytes_ge<BQ_HI>(v.x, t_low) & ~drop.x, l1 = bytes_ge<BQ_HI>(v.y, t_low) & ~drop.y;
    const uint32_t l2 = bytes_ge<BQ_HI>(v.z, t_low) & ~drop.z, l3 = bytes_ge<BQ_HI>(v.w, t_low) & ~drop.w;
    acc = __dp4a(v.x, l0, __dp4a(v.y, l1, __dp4a(v.z, l2, __dp4a(v.w, l3, acc))));
    red_shared(dst, l0 >> 7); red_shared(dst + 4, l1 >> 7); red_shared(dst + 8, l2 >> 7); red_shared(dst + 12, l3 >> 7);
}

// Stream one M-segment: qs = byte offset of its first quality inside the stage (the stage keeps the 16-byte phase of
// the global column), len bases, rrel = window entry of the first base.  Entry e of class a lives at byte e + 16 - a of
// array a, so a chunk whose byte 0 is entry e0 adds its four words to words (e0 >> 2) + 4 .. + 7 of array e0 & 3.
// A segment of two or more chunks needs one mask for its first chunk (bytes below head) and one for its last.
template <bool BQ_HI>
__device__ __forceinline__ void stream_segment(uint32_t stage_s, uint32_t sC_s, uint32_t qs, uint32_t len, uint32_t rrel,
                                               const uint4 *sMaskLo, const uint4 *sMaskHi, uint32_t t_low, uint32_t &acc) {
    const uint4 none = make_uint4(0, 0, 0, 0);
    const uint32_t head = qs & 15u;
    const uint32_t nc = (head + len + 15u) >> 4;
    uint32_t src = stage_s + (qs & ~15u);
    const int e0 = (int)rrel - (int)head;                                  // >= -15
    uint32_t dst = sC_s + ((uint32_t)e0 & 3u) * (uint32_t)(F_CW * 4) + (uint32_t)(((e0 >> 2) + 4) * 4);
    if (nc == 1u) { count_words<BQ_HI>(lds128(src), or4(sMaskLo[head], sMaskHi[head + len]), dst, t_low, acc); return; }
    count_words<BQ_HI>(lds128(src), sMaskLo[head], dst, t_low, acc);
    uint32_t n_int = nc - 2u;                                              // interior chunks: no masks
    src += 16; dst += 16;
#pragma unroll 1
    for (; n_int >= 2u; n_int -= 2u) {
        const uint4 v0 = lds128(src), v1 = lds128(src + 16);               // both loads in flight before the first count
        count_words<BQ_HI>(v0, none, dst, t_low, acc); count_words<BQ_HI>(v1, none, dst + 16, t_low, acc);
        src += 32; dst += 32;
    }
    if (n_int) { count_words<BQ_HI>(lds128(src), none, dst, t_low, acc); src += 16; dst += 16; }
    count_words<BQ_HI>(lds128(src), sMaskHi[head + len - 16u * (nc - 1u)], dst, t_low, acc);
}

// Same from global memory (the few second-and-later M-segments of a window: their qualities are in L2, one 16-byte
// load per chunk; src0 = 16-byte aligned address of the window's first quality byte, qs relative to it).
template <bool BQ_HI>
__device__ __forceinline__ void stream_segment_global(const uint8_t *src0, uint32_t sC_s, uint32_t qs, uint32_t len, uint32_t rrel,
                                                      const uint4 *sMaskLo, const uint4 *sMaskHi, uint32_t t_low, uint32_t &acc,
                                                      uint32_t c_first, uint32_t c_step, const uint8_t *q_lo, const uint8_t *q_hi) {
    const uint32_t head = qs & 15u;
    const uint32_t nc = (head + len + 15u) >> 4;
    const uint4 *src = reinterpret_cast<const uint4 *>(src0 + (qs & ~15u));
    const int e0 = (int)rrel - (int)head;
    const uint32_t dst0 = sC_s + ((uint32_t)e0 & 3u) * (uint32_t)(F_CW * 4) + (uint32_t)(((e0 >> 2) + 4) * 4);
#pragma unroll 1
    for (uint32_t c = c_first; c < nc; c += c_step) {              // the caller spreads the chunks of a segment over c_step threads
        if (!CLB_GMEM_OK(src + c, q_lo, q_hi)) continue;
        const uint32_t lo = c == 0 ? head : 0u, hi = min(16u, head + len - 16u * c);
        count_words<BQ_HI>(ldg_stream(src + c), or4(sMaskLo[lo], sMaskHi[hi]), dst0 + 16u * c, t_low, acc);
    }
}

// What a thread knows about its read of the next sub-batch: loaded one sub-batch ahead so that the DRAM round trips
// overlap the streaming of the current one.
struct FMeta {
    int ps, pback; uint32_t fl, mq, c0, c1, op0, op1, op2, q0, q1;   // q0, q1: relative to the window's first quality byte
};
// the first three CIGAR ops in one round trip (almost every short read has at most three)
__device__ __forceinline__ void fmeta_ops(const KParams &P, FMeta &M) {
    M.op0 = M.c1 > M.c0 ? P.cigar[M.c0] : 0xfu;
    M.op1 = M.c1 > M.c0 + 1u ? P.cigar[M.c0 + 1u] : 0xfu;
    M.op2 = M.c1 > M.c0 + 2u ? P.cigar[M.c0 + 2u] : 0xfu;
}
__device__ __forceinline__ void fmeta_load(const KParams &P, FMeta &M, uint32_t ic, uint64_t wqx) {
    M.fl = P.flag[ic]; M.c0 = P.cigar_off[ic]; M.c1 = P.cigar_off[ic + 1];
    M.ps = P.pos[ic]; M.mq = P.mapq[ic];
    M.q0 = (uint32_t)(P.qual_off[ic] - wqx); M.q1 = (uint32_t)(P.qual_off[ic + 1] - wqx);   // k_window_ranges checked the window's range fits 32 bits
    M.pback = P.pos[ic >= (uint32_t)F_LOOKBACK ? ic - (uint32_t)F_LOOKBACK : 0u];
}

template <bool BQ_HI, bool DBG, unsigned FEAT = 0u>
__global__ void __launch_bounds__(NT, CLB_F_MINB) k_pileup_fast(const KParams P) {
    constexpr bool HIST = (FEAT & FEAT_HIST) != 0, TILES = (FEAT & FEAT_TILES) != 0, RUNS = (FEAT & FEAT_RUNS) != 0;
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const uint32_t w = P.win_first + blockIdx.x;
    // one table record per window, three independent 16-byte loads (no dependent round trip)
    const uint4 wg = P.win_rec[3 * (size_t)w + 2];                         // x: reads per sub-batch (0: general-path window)
    const uint4 wr = P.win_rec[3 * (size_t)w];
    const ulonglong2 wq = *reinterpret_cast<const ulonglong2 *>(P.win_rec + 3 * (size_t)w + 1);
    const uint32_t G = wg.x;
    if (G == 0) return;
    if (*P.err & ERR_INPUT_REFUSED) return;                                // do not walk refused columns
    CLB_STAMP(0);

    uint32_t *sA = reinterpret_cast<uint32_t *>(smem_raw + F_OFF_A);
    uint32_t *sC = reinterpret_cast<uint32_t *>(smem_raw + F_OFF_C);
    uint2 *sX = reinterpret_cast<uint2 *>(smem_raw + F_OFF_X);
    const uint4 *sMaskLo = reinterpret_cast<const uint4 *>(smem_raw + F_OFF_MASK);
    const uint4 *sMaskHi = sMaskLo + 17;
    const uint8_t *sFirst = smem_raw + F_OFF_FIRST;
    uint32_t *sScan = reinterpret_cast<uint32_t *>(smem_raw + F_OFF_SCAN);
    uint8_t *sLast = smem_raw + F_OFF_LAST;
    unsigned long long *sWStats = reinterpret_cast<unsigned long long *>(smem_raw + F_OFF_WSTATS);
    volatile uint32_t *sCtl = reinterpret_cast<volatile uint32_t *>(smem_raw + F_OFF_CTL);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t sA_s = smem_addr(sA), sC_s = smem_addr(sC);
    const uint32_t stage_s = smem_addr(smem_raw + F_OFF_STAGE) + (uint32_t)warp * F_WSTAGE;   // this warp's stage
    const uint32_t bar = smem_addr(smem_raw + F_OFF_BAR) + 8u * (uint32_t)warp;                // and its mbarrier
    const uint32_t xcnt_s = smem_addr(const_cast<uint32_t *>(&sCtl[FC_XCNT]));

    const uint32_t wb0 = P.region_start + w * (uint32_t)WREAL;                           // position of entry 0 (BAM positions are below 2^31)
    const uint32_t n_ent = min((uint32_t)WREAL, P.region_end - wb0);                     // entries in use, 1 .. WREAL
    const uint32_t r_lo = wr.x, r_hi = wr.y;
    const uint32_t n_sub = wg.y;                                           // = ceil((r_hi - r_lo) / G), divided once by k_window_ranges;                     // sub-batches of G <= 32 reads; warp v takes v, v + 8, ...
    const uint32_t ebase = tid * PPT;

    // loads whose latency the setup hides: this warp's first sub-batch and the REF_N bits of phase C
    FMeta M;
    uint32_t j = (uint32_t)warp;
    if (j < n_sub) fmeta_load(P, M, min(r_lo + j * G + (uint32_t)lane, r_hi - 1u), wq.x);
    uint32_t nm0, nm1;
    {
        const uint32_t p0 = wb0 + ebase;
        nm0 = P.nmask[p0 >> 5]; nm1 = P.nmask[(p0 >> 5) + 1];
    }
    const uint32_t max_span = r_hi > r_lo ? *P.max_span : 0u;
    // the CIGAR ops are the last hop of the window's first dependent chain (table record -> columns -> ops): start them towards L2 now
    if (tid == 0 && wg.w > wg.z) l2_prefetch(P.cigar, 4ull * wg.z, 4ull * wg.w, 64u << 10);
    {
        uint4 *z = reinterpret_cast<uint4 *>(smem_raw);
        for (int i = tid; i < (F_OFF_STAGE / 16); i += NT) z[i] = make_uint4(0, 0, 0, 0);
        const uint4 *msrc = reinterpret_cast<const uint4 *>(P.win_tables);               // byte masks (first 2 x 17 x 16 bytes)
        uint4 *mdst = reinterpret_cast<uint4 *>(smem_raw + F_OFF_MASK);
        if (tid < 34) mdst[tid] = msrc[tid];
        const uint4 *fsrc = reinterpret_cast<const uint4 *>(P.first_tab8);
        uint4 *fdst = reinterpret_cast<uint4 *>(smem_raw + F_OFF_FIRST);
        if (tid >= 64 && tid < 64 + F_NFIRST / 16) fdst[tid - 64] = fsrc[tid - 64];
        if (tid < 4) sCtl[tid] = 0;
        if (lane == 0) mbar_init(bar, 1);
    }
    __syncthreads();
    CLB_STAMP(1);
    if (j < n_sub) fmeta_ops(P, M);

    const uint32_t t_low = (P.min_bq & 0x7fu) * 0x01010101u;
    const uint32_t min_mapq = P.min_mapq, max_low_mapq = P.max_low_mapq;
    uint32_t acc128 = 0;                                                   // 128 x sum of passing qualities of the current sub-batch
    // sums of one window fit 32 bits: at most 2047 positions x 254 reads (depth proof) x 255
    uint32_t acc_sum = 0, acc_mapq = 0;
    uint32_t parity = 0;

    // Every warp runs its own pipeline: bulk copy of its sub-batch's qualities -> CIGAR walk while the copy is in
    // flight -> next sub-batch's columns requested -> wait for the copy -> stream.  Only __syncwarp inside.
    for (; j < n_sub; j += NWARPS) {
        const uint32_t rb = r_lo + j * G, n = min(G, r_hi - rb);
        __syncwarp();                                                      // every lane is done with the stage
        const uint32_t q_first = __shfl_sync(FULL, M.q0, 0), q_last = __shfl_sync(FULL, M.q1, (int)n - 1);
        const uint32_t sb = q_first & ~15u;                                // stage byte 0 <-> this byte of the window's qualities (wq.x is 16-byte aligned)
        const uint32_t bytes = (q_last - sb + 15u) & ~15u;                 // q_last <= 0xfffffff0: no wrap
        const bool fits = bytes <= (uint32_t)F_WSTAGE;                     // k_window_ranges sized the sub-batches: always true
        if (!fits) sCtl[FC_BAIL] = 1;
        if (lane == 0 && fits && bytes) { mbar_arrive_expect_tx(bar, bytes); bulk_g2s(stage_s, P.qual + wq.x + sb, bytes, bar); }

        // ---------------------------------------------------------------- phase A: one read per lane
        bool has0 = false; uint32_t s_qs = 0, s_len = 0, s_rr = 0;
        {
            const bool valid = (uint32_t)lane < n;
            const bool live = valid && !(M.fl & 4u) && M.c1 > M.c0;
            uint32_t nops = live ? M.c1 - M.c0 : 0u;
            const uint32_t ic = rb + (uint32_t)lane;
            const bool deep = valid && ic >= (uint32_t)F_LOOKBACK && (long long)M.pback + (long long)max_span > (long long)M.ps;
            if (deep || nops > (uint32_t)F_MAXOPS) { sCtl[FC_BAIL] = 1; nops = 0; }
            const uint32_t lq = M.q1 - M.q0;
            const uint32_t qs_base = M.q0 - sb;                            // offset of the read's first quality inside the stage
            const uint32_t qx_base = M.q0;                                 // ... and relative to the window's first quality byte
            const int rel = M.ps - (int)wb0;
            const uint32_t mq = M.mq, c0 = M.c0;
            const bool pass = mq >= min_mapq;
            const uint32_t kmax = __reduce_max_sync(FULL, nops);
            int rp = rel; uint32_t qp = 0;
            for (uint32_t k = 0; k < kmax; k++) {
                uint32_t v = k == 0 ? M.op0 : k == 1 ? M.op1 : M.op2;
                if (k >= 3u && k < nops) v = P.cigar[c0 + k];
                if (k >= nops) v = 0xfu;                                                   // op 15, len 0: no effect (skipped reads, shorter CIGARs)
                const uint32_t op = v & 15u, len = v >> 4;
                if (((0x181u >> op) & 1u) && pass && qp < lq && rp < (int)n_ent) {          // M, =, X with qualities, not right of the window
                    const uint32_t l = min(len, lq - qp);
                    const int s = max(rp, 0);
                    const int e = min(rp + (int)l, (int)n_ent);                            // rp < 2048, l < 2^28: no overflow
                    if (e > s) {
                        const uint32_t qo = qp + (uint32_t)(s - rp);
                        if (!has0) { has0 = true; s_qs = qs_base + qo; s_len = (uint32_t)(e - s); s_rr = (uint32_t)s; }
                        else {
                            const uint32_t idx = atom_shared_add(xcnt_s, 1u);
                            if (idx < (uint32_t)F_XCAP) sX[idx] = make_uint2(qx_base + qo, (uint32_t)s | ((uint32_t)(e - s) << 11));
                            else sCtl[FC_BAIL] = 1;
                        }
                    }
                }
                if (((0x18du >> op) & 1u) && rp < (int)WN) rp += (int)len;                  // M, D, N, =, X consume the reference
                if ((0x193u >> op) & 1u) qp += len;                                         // M, I, S, =, X consume the query
            }
            if (nops) {
                const int s = max(rel, 0), e = min(rp, (int)n_ent);
                if (e > s) {
                    const uint32_t delta = 1u + (mq <= max_low_mapq ? 0x10000u : 0u);       // raw depth | low-MAPQ depth << 16
                    red_shared(sA_s + 4u * (uint32_t)s, delta);
                    red_shared(sA_s + 4u * (uint32_t)e, 0u - delta);                        // e <= n_ent <= WREAL < WN
                    if (pass) acc_mapq += mq * (uint32_t)(e - s);
                }
            }
        }
        // this warp's next sub-batch: its columns are in flight while the current one is streamed
        if (j == 0) CLB_STAMP(2);
        const bool has_next = j + NWARPS < n_sub;
        if (has_next) fmeta_load(P, M, min(r_lo + (j + NWARPS) * G + (uint32_t)lane, r_hi - 1u), wq.x);
        if (fits && bytes) { mbar_wait(bar, parity); parity ^= 1u; }       // the staged qualities have landed
        if (j == 0) CLB_STAMP(3);
        if (has_next) fmeta_ops(P, M);
        // ---------------------------------------------------------------- phase B: stream from shared memory
        if (has0 && fits) stream_segment<BQ_HI>(stage_s, sC_s, s_qs, s_len, s_rr, sMaskLo, sMaskHi, t_low, acc128);
        if (j == 0) CLB_STAMP(4);
        acc_sum += acc128 >> 7; acc128 = 0;                                // at most 2047 bases x 255 x 128 per sub-batch: no overflow
    }
    __syncthreads();                                                       // every warp's pushes / counters
    if (sCtl[FC_BAIL]) {
        // not an ordinary window after all: hand it to the general kernel (nothing global was written yet)
        if (tid == 0) P.gen_list[atomicAdd(P.gen_count, 1u)] = w;
        return;
    }
    {
        // second-and-later M-segments of the window's reads (indels): few, pooled for the whole CTA, streamed from L2
        const uint32_t nx = sCtl[FC_XCNT];
        if (nx) {
            for (uint32_t x = (uint32_t)tid >> 4; x < nx; x += NT / 16) {  // 16 threads per segment, one chunk each: one L2 round trip
                const uint2 d = sX[x];
                stream_segment_global<BQ_HI>(P.qual + wq.x, sC_s, d.x, d.y >> 11, d.y & 0x7ffu, sMaskLo, sMaskHi, t_low, acc128,
                                             (uint32_t)tid & 15u, 16u, P.qual, P.qual + P.qual_bytes);
            }
            acc_sum += acc128 >> 7;
            __syncthreads();
        }
    }

    CLB_STAMP(5);
    // ------------------------------------------------------------------ phase C: scan, classify, segment
    static_assert(PPT == 8, "phase C of the fast kernel is written for 8 entries per thread");
    // The stages are dead since the barrier after the main loop (each warp's last sub-batch has streamed) and nothing has
    // gone to global memory (a window that bailed returned above): zero the depth table here, the scan barrier below orders
    // it before the first count.
    uint32_t *sHist = reinterpret_cast<uint32_t *>(smem_raw + F_OFF_HIST);
    if constexpr (HIST) zero_depth_table(sHist);
    uint32_t a[PPT], qcv[PPT];
    {
        const uint4 a0 = *reinterpret_cast<const uint4 *>(sA + ebase), a1 = *reinterpret_cast<const uint4 *>(sA + ebase + 4);
        a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w; a[4] = a1.x; a[5] = a1.y; a[6] = a1.z; a[7] = a1.w;
        // qc depth: entries ebase .. ebase + 7 are bytes ebase + 16 - cls .. of class array cls
        const uint32_t W = 2u * (uint32_t)tid + 4u;
        const uint2 c0v = *reinterpret_cast<const uint2 *>(sC + W);
        uint32_t lo = c0v.x, hi = c0v.y;
#pragma unroll
        for (int cls = 1; cls < 4; cls++) {
            const uint32_t *row = sC + cls * F_CW + W;
            const uint32_t wm = row[-1];
            const uint2 wv = *reinterpret_cast<const uint2 *>(row);
            lo += __funnelshift_r(wm, wv.x, 8u * (4u - (uint32_t)cls));
            hi += __funnelshift_r(wv.x, wv.y, 8u * (4u - (uint32_t)cls));
        }
        qcv[0] = lo & 0xffu; qcv[1] = (lo >> 8) & 0xffu; qcv[2] = (lo >> 16) & 0xffu; qcv[3] = lo >> 24;
        qcv[4] = hi & 0xffu; qcv[5] = (hi >> 8) & 0xffu; qcv[6] = (hi >> 16) & 0xffu; qcv[7] = hi >> 24;
    }
#pragma unroll
    for (int k = 1; k < PPT; k++) a[k] += a[k - 1];
    {
        const uint32_t ta = a[PPT - 1];
        uint32_t ia = ta;
#pragma unroll
        for (int dd = 1; dd < 32; dd <<= 1) { const uint32_t t1 = __shfl_up_sync(FULL, ia, dd); if (lane >= dd) ia += t1; }
        if (lane == 31) sScan[warp] = ia;
        __syncthreads();
        const uint32_t oa = ia - ta + __reduce_add_sync(FULL, lane < warp ? sScan[lane] : 0u);
#pragma unroll
        for (int k = 0; k < PPT; k++) a[k] += oa;
    }
    const uint32_t nbits = __funnelshift_r(nm0, nm1, (wb0 + ebase) & 31u);
    Entries<uint32_t> e = entries_of<uint32_t>(ebase, 0u, n_ent);          // no halo entry
    const StateLimits lim = state_limits(P);
    DepthHist dh{};
    if constexpr (HIST) dh = depth_hist_of(smem_addr(sHist), P);
#pragma unroll
    for (int k = 0; k < PPT; k++) {
        const uint32_t raw = a[k] & 0xffffu;
        classify_entry(e, k, raw, a[k] >> 16, qcv[k], sFirst[raw], (nbits >> k) & 1u, lim);   // one byte per depth: raw <= 254 (depth proof)
        if constexpr (HIST) count_depth<true>(dh, e, k, raw, qcv[k]);      // qc <= raw <= 254: the table holds every depth
    }
    if constexpr (HIST) close_depth_runs<true>(dh);
    close_entries(e, n_ent, sLast, sScan);
    const auto raw_of = [&](int k) { return a[k] & 0xffffu; };            // not the packed word: its high half is the low-MAPQ depth
    uint32_t *sRunLast = reinterpret_cast<uint32_t *>(smem_raw + F_OFF_RUN);
    if constexpr (RUNS) publish_run_depth(e, n_ent, raw_of, sRunLast, sScan);
    dbg_dump<DBG>(e, w * (uint32_t)WREAL, [&](int k) { return make_uint3(a[k] & 0xffffu, qcv[k], a[k] >> 16); }, P);
    unsigned long long *sTileSum = reinterpret_cast<unsigned long long *>(smem_raw + F_OFF_TILE);
    uint32_t *sTileFirst = reinterpret_cast<uint32_t *>(sTileSum + NWARPS * 8);
    if constexpr (TILES) count_tiles(e, wb0, nbits, [&](int k) { return make_uint2(a[k] & 0xffffu, qcv[k]); }, sTileSum, sTileFirst, P);
    reduce_stats(e, acc_sum, acc_mapq, sWStats, P);
    if constexpr (HIST) flush_depth_table(dh, sHist);                      // after reduce_stats' barrier
    if constexpr (TILES) flush_tiles(sTileSum, sTileFirst, P);
    // the window's first position always starts a record and a depth run (window soft: the gather drops them when the
    // previous window ended in the same state / at the same raw depth)
    const uint32_t rmask = RUNS ? run_starts(e, raw_of, 0u, sRunLast) : 0u;
    write_records<RUNS>(e, wb0, 0u, 0u, w > 0 ? 1u : 0u, sLast, sScan, w, P, rmask, raw_of);
    add_bins(e, wb0, 0u, n_ent, wr.z, wr.w - 1u, P);                       // k_window_ranges counts the next bin's entry from the halo
    CLB_STAMP(6);
    CLB_STAMP_VALUE(7, r_hi - r_lo);
}

}  // namespace clb
