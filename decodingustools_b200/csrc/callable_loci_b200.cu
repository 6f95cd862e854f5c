// callable_loci_b200.cu -- C-ABI implementation (device path) of include/callable_loci_b200.h.
//
// Host orchestration of the sm_100a kernels in clb_kernels.cuh: device buffers for the packed read
// columns, double-stream copy/compute overlap (column batches are copied on one stream while the
// windows they complete run on another), interval compaction and the device->host result copy.
// Reference seam replaced: callable_loci::process_single_contig, /root/reference/src/callable_loci/mod.rs:44-147.
#include "../../include/callable_loci_b200.h"
#include "clb_kernels.cuh"
#include "clb_fast.cuh"

#include <dlfcn.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

using namespace clb;

namespace {

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;   // bytes
};

struct EvPair { cudaEvent_t a, b; };

}  // namespace

struct clb_ctx {
    int device = 0;
    clb_options opt{};
    std::string err;
    cudaStream_t s_own = nullptr, s_copy = nullptr, s_compute = nullptr;
    cudaEvent_t ev_copy = nullptr;
    std::vector<EvPair> ev_pool;        // reusable timing event pairs
    std::vector<EvPair> ev_kernel, ev_h2d, ev_upload;
    uint32_t *d_first_tab = nullptr;
    int max_ctas_per_sm = 0, n_sm = 0;
    bool force_general = false;         // CLB_FORCE_GENERAL=1: every window through the general kernel (A/B measurements, tests)

    // contig state
    bool in_contig = false, finished = false;
    int32_t tid = 0;
    std::string name;
    uint32_t contig_len = 0, largest = 0, region_start = 0, region_end = 0;
    uint32_t n_windows = 0, windows_done = 0;
    uint32_t stride = 0, n_bins = 0;
    uint32_t dh_next = 0, dh_n = 0;     // depth-histogram bins: set by clb_set_depth_histogram, in force for the current contig
    uint32_t dh_fetched = 0;            // ... and in the result of the last fetch (clb_depth_histogram)
    uint32_t tl_next = 0, tl_len = 0;   // depth-tile length: set by clb_set_depth_tiles, in force for the current contig
    uint32_t n_tiles = 0;               // ceil(contig_len / tl_len) while on
    uint32_t tl_fetched = 0;            // tiles in the result of the last fetch (clb_depth_tiles)
    bool runs_next = false, runs = false;   // depth runs: set by clb_set_depth_runs, in force for the current contig
    bool runs_fetched = false;              // ... and in the result of the last fetch (clb_depth_runs)
    bool long_mode = false, span_on_device = false;
    uint64_t n_reads = 0, n_cigar = 0, n_qual = 0;
    long long last_pos = -1;

    DevBuf pos, flag, mapq, cigar_off, cigar, qual_off, qual, read_end, cigar_ckpt;
    DevBuf nmask, ref_ascii;
    DevBuf stats_padded, counters, rec, win_tab, win_rec, win_out, deep_list, intervals, misc;
    DevBuf gen_list, blk_tot, dhist;
    DevBuf run_rec, run_win_tab, runs_out;   // depth runs: records, window table, compacted runs (region length each)
    DevBuf dbg_raw, dbg_qc, dbg_low, dbg_state, timing;
    uint32_t rec_cap = 0;
    bool dbg = false;

    // host-side result storage
    clb_interval *h_intervals = nullptr;   // pinned
    size_t h_intervals_cap = 0;
    std::vector<unsigned long long> h_counters;
    std::vector<uint32_t> h_bins;
    uint32_t *h_misc = nullptr;            // pinned mirror of misc
    uint64_t h2d_bytes = 0, d2h_bytes = 0;
    uint32_t launches = 0;
    uint64_t n_intervals = 0;
    clb_depth_run *h_runs = nullptr;       // pinned
    size_t h_runs_cap = 0;
    uint64_t n_runs = 0;
};

// misc layout (uint32): record cursor, error bits, n_total intervals, deep-window count, general-queue count / tickets taken
// (these six are reset per run), then the maximum reference span; with depth runs on, the run cursor and run count follow
// (reset per run too, and only copied then)
enum { M_CURSOR = 0, M_ERR = 1, M_NTOTAL = 2, M_DEEP = 3, M_GEN_COUNT = 4, M_GEN_TAKEN = 5, M_RESET_WORDS = 6, M_MAXSPAN = 7, M_MAXQLEN = 8, M_WORDS = 9,
       M_RUN_CURSOR = 9, M_RUN_NTOTAL = 10, M_WORDS_RUNS = 11 };

namespace {

int fail(clb_ctx *c, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
    if (c) c->err = buf;
    return code;
}

#define CU(call)                                                                                              \
    do {                                                                                                      \
        cudaError_t e_ = (call);                                                                              \
        if (e_ != cudaSuccess) return fail(ctx, CLB_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

int ensure(clb_ctx *ctx, DevBuf &b, size_t bytes, bool keep, cudaStream_t s) {
    if (bytes <= b.cap) return CLB_OK;
    size_t ncap = std::max(bytes, keep ? b.cap + b.cap / 2 : (size_t)0);
    ncap = (ncap + 255) & ~(size_t)255;
    void *np = nullptr;
    CU(cudaMalloc(&np, ncap));
    if (b.p) {
        if (keep) {
            // kernels of earlier windows may still read the old buffer: drain both streams first
            CU(cudaStreamSynchronize(ctx->s_compute));
            CU(cudaStreamSynchronize(ctx->s_copy));
            CU(cudaMemcpyAsync(np, b.p, b.cap, cudaMemcpyDeviceToDevice, s));
            CU(cudaStreamSynchronize(s));
        } else {
            CU(cudaStreamSynchronize(ctx->s_compute));
            CU(cudaStreamSynchronize(ctx->s_copy));
        }
        CU(cudaFree(b.p));
    }
    b.p = np; b.cap = ncap;
    return CLB_OK;
}

void release(DevBuf &b) { if (b.p) cudaFree(b.p); b.p = nullptr; b.cap = 0; }

// u64 words of the counter buffer: [N_STATS stats][3 x n_bins bins][n raw][n qc][territory T][callable T][raw_sum T][qc_sum T]
// (histograms and tiles only when on)
size_t tiles_offset(const clb_ctx *c) { return (size_t)N_STATS + 3 * (size_t)c->n_bins + 2 * (size_t)c->dh_n; }
size_t n_counters(const clb_ctx *c) { return tiles_offset(c) + 4 * (size_t)c->n_tiles; }

int get_events(clb_ctx *ctx, EvPair &ep) {
    if (!ctx->ev_pool.empty()) { ep = ctx->ev_pool.back(); ctx->ev_pool.pop_back(); return CLB_OK; }
    CU(cudaEventCreate(&ep.a)); CU(cudaEventCreate(&ep.b));
    return CLB_OK;
}

KParams make_params(clb_ctx *c) {
    KParams P{};
    P.pos = (const int32_t *)c->pos.p; P.flag = (const uint16_t *)c->flag.p; P.mapq = (const uint8_t *)c->mapq.p;
    P.cigar_off = (const uint32_t *)c->cigar_off.p; P.cigar = (const uint32_t *)c->cigar.p;
    P.qual_off = (const uint64_t *)c->qual_off.p; P.qual = (const uint8_t *)c->qual.p; P.qual_bytes = c->qual.cap;
    P.read_end = c->long_mode ? (const uint32_t *)c->read_end.p : nullptr;
    P.cigar_ckpt = c->long_mode ? (const uint2 *)c->cigar_ckpt.p : nullptr;
    P.nmask = (const uint32_t *)c->nmask.p;
    P.region_start = c->region_start; P.region_end = c->region_end;
    P.min_depth = c->opt.min_depth; P.max_depth = c->opt.max_depth; P.min_depth_for_low_mapq = c->opt.min_depth_for_low_mapq;
    P.min_mapq = c->opt.min_mapping_quality; P.min_bq = c->opt.min_base_quality; P.max_low_mapq = c->opt.max_low_mapq;
    P.first_tab = c->d_first_tab;
    P.win_tables = c->d_first_tab + 65536;
    P.first_tab8 = (const uint8_t *)(c->d_first_tab + 65536) + WIN_TABLE_BYTES;
    P.win_rec = (const uint4 *)c->win_rec.p;
    P.stats = (unsigned long long *)c->stats_padded.p;
    P.bins = (unsigned long long *)c->counters.p + N_STATS;
    P.n_bins = c->n_bins; P.stride = c->stride;
    P.rec = (unsigned long long *)c->rec.p; P.rec_cap = c->rec_cap;
    P.rec_cursor = (uint32_t *)c->misc.p + M_CURSOR;
    P.win_tab = (uint2 *)c->win_tab.p;
    P.err = (uint32_t *)c->misc.p + M_ERR;
    P.deep_count = (uint32_t *)c->misc.p + M_DEEP; P.deep_list = (uint32_t *)c->deep_list.p;
    P.gen_list = (uint32_t *)c->gen_list.p;
    P.gen_count = (uint32_t *)c->misc.p + M_GEN_COUNT; P.gen_taken = (uint32_t *)c->misc.p + M_GEN_TAKEN;
    P.max_span = (const uint32_t *)c->misc.p + M_MAXSPAN;
    P.max_low_mapq_fraction = c->opt.max_low_mapq_fraction;
    P.timing = (long long *)c->timing.p;
    P.dhist = c->dh_n ? (unsigned long long *)c->dhist.p : nullptr; P.dh_n = c->dh_n;
    P.tiles = c->tl_len ? (unsigned long long *)c->counters.p + tiles_offset(c) : nullptr; P.tile_len = c->tl_len; P.n_tiles = c->n_tiles;
    if (c->runs) {
        P.run_rec = (uint2 *)c->run_rec.p; P.run_cursor = (uint32_t *)c->misc.p + M_RUN_CURSOR; P.run_win_tab = (uint4 *)c->run_win_tab.p;
        P.run_cap = c->region_end - c->region_start;
    }
    if (c->dbg) {
        P.dbg_raw = (uint32_t *)c->dbg_raw.p; P.dbg_qc = (uint32_t *)c->dbg_qc.p;
        P.dbg_low = (uint32_t *)c->dbg_low.p; P.dbg_state = (uint8_t *)c->dbg_state.p;
    }
    return P;
}

// The pileup kernels' template arguments: BQ_HI = (min_base_quality >= 128) picks the byte compare, DBG the instantiation
// with the per-base dump (parity tests), FEAT the optional outputs that are on (FEAT_HIST: depth histograms, FEAT_TILES:
// depth tiles, FEAT_RUNS: depth runs; only launched when on, so the others stay as they were).  f is called with two
// std::integral_constant<bool, ...> and one std::integral_constant<unsigned, FEAT>.
template <unsigned X> using FeatC = std::integral_constant<unsigned, X>;
template <typename F>
void with_variant(bool bq_hi, bool dbg, unsigned feat, F &&f) {
    using T = std::true_type; using N = std::false_type;
    auto h = [&](auto b, auto d) {
        switch (feat) {
        case 0: f(b, d, FeatC<0u>{}); break;
        case 1: f(b, d, FeatC<1u>{}); break;
        case 2: f(b, d, FeatC<2u>{}); break;
        case 3: f(b, d, FeatC<3u>{}); break;
        case 4: f(b, d, FeatC<4u>{}); break;
        case 5: f(b, d, FeatC<5u>{}); break;
        case 6: f(b, d, FeatC<6u>{}); break;
        default: f(b, d, FeatC<7u>{}); break;
        }
    };
    if (bq_hi) { if (dbg) h(T{}, T{}); else h(T{}, N{}); }
    else { if (dbg) h(N{}, T{}); else h(N{}, N{}); }
}
unsigned features(const clb_ctx *c) { return (c->dh_n ? FEAT_HIST : 0u) | (c->tl_len ? FEAT_TILES : 0u) | (c->runs ? FEAT_RUNS : 0u); }

// window ranges + classes, the fast kernel (one CTA per window) and the general kernel (persistent CTAs over the
// queue of windows the other two handed over) for windows [w0, w1) on the compute stream
int launch_windows(clb_ctx *ctx, uint32_t w0, uint32_t w1, EvPair *time_pileup = nullptr, EvPair *time_fast = nullptr) {
    if (w1 <= w0) return CLB_OK;
    const uint32_t n = w1 - w0;
    const bool all_general = ctx->force_general || ctx->long_mode;
    k_window_ranges<<<(unsigned)(((uint64_t)n * WR_LANES + 255) / 256), 256, 0, ctx->s_compute>>>(   // WR_LANES lanes per window
        (const int32_t *)ctx->pos.p, (uint32_t)ctx->n_reads, ctx->region_start, ctx->region_end,
        (const uint32_t *)ctx->misc.p + M_MAXSPAN, w0, n, (const uint64_t *)ctx->qual_off.p, (const uint32_t *)ctx->cigar_off.p, ctx->stride,
        (uint4 *)ctx->win_rec.p, all_general ? 1u : 0u, (uint32_t *)ctx->gen_list.p, (uint32_t *)ctx->misc.p + M_GEN_COUNT,
        (const uint32_t *)ctx->misc.p + M_MAXQLEN);
    KParams P = make_params(ctx);
    P.win_first = w0;
    if (time_pileup) CU(cudaEventRecord(time_pileup->a, ctx->s_compute));
    const bool hi = ctx->opt.min_base_quality >= 128;
    if (!all_general) {
        if (time_fast) CU(cudaEventRecord(time_fast->a, ctx->s_compute));
        with_variant(hi, ctx->dbg, features(ctx), [&](auto h, auto d, auto x) {
            k_pileup_fast<decltype(h)::value, decltype(d)::value, decltype(x)::value><<<n, NT, F_SMEM, ctx->s_compute>>>(P);
        });
        if (time_fast) CU(cudaEventRecord(time_fast->b, ctx->s_compute));
        ctx->launches += 1;
    }
    const uint32_t g = (uint32_t)std::min<uint64_t>((uint64_t)ctx->n_sm * std::max(1, ctx->max_ctas_per_sm), all_general ? n : 0xffffffffu);
    with_variant(hi, ctx->dbg, features(ctx), [&](auto h, auto d, auto x) {
        k_pileup_general<decltype(h)::value, decltype(d)::value, decltype(x)::value><<<g, NT, SMEM_BYTES, ctx->s_compute>>>(P);
    });
    if (time_pileup) CU(cudaEventRecord(time_pileup->b, ctx->s_compute));
    ctx->launches += 2;
    CU(cudaGetLastError());
    return CLB_OK;
}

int reset_accumulators(clb_ctx *ctx) {
    CU(cudaMemsetAsync(ctx->stats_padded.p, 0, (size_t)N_STATS * STAT_STRIDE * 8, ctx->s_compute));
    CU(cudaMemsetAsync(ctx->counters.p, 0, n_counters(ctx) * 8, ctx->s_compute));
    if (ctx->dh_n) CU(cudaMemsetAsync(ctx->dhist.p, 0, (size_t)DH_SLOTS * 2 * ctx->dh_n * 8, ctx->s_compute));
    CU(cudaMemsetAsync((uint32_t *)ctx->misc.p + M_CURSOR, 0, M_RESET_WORDS * sizeof(uint32_t), ctx->s_compute));   // cursor, err, n_total, deep windows, general queue
    if (ctx->runs) CU(cudaMemsetAsync((uint32_t *)ctx->misc.p + M_RUN_CURSOR, 0, 2 * sizeof(uint32_t), ctx->s_compute));   // run cursor, run count
    return CLB_OK;
}

int launch_compaction(clb_ctx *ctx) {
    if (ctx->n_windows == 0) return CLB_OK;
    {
        // windows with more than 65535 candidate reads were queued by the general kernel (normally none)
        const KParams P = make_params(ctx);
        with_variant(ctx->opt.min_base_quality >= 128, ctx->dbg, features(ctx), [&](auto h, auto d, auto x) {
            k_pileup_classify_deep<decltype(h)::value, decltype(d)::value, decltype(x)::value><<<ctx->n_sm, NT, SMEM_BYTES_DEEP, ctx->s_compute>>>(P);
        });
        ctx->launches += 1;
    }
    const uint32_t n_blk = (ctx->n_windows + 1023) / 1024;
    k_scan_windows_local<uint2><<<n_blk, 1024, 0, ctx->s_compute>>>((const uint2 *)ctx->win_tab.p, ctx->n_windows, (uint32_t *)ctx->win_out.p,
                                                            (uint32_t *)ctx->blk_tot.p, (const uint32_t *)ctx->misc.p + M_ERR);
    k_scan_blocks<<<1, 1024, 0, ctx->s_compute>>>((uint32_t *)ctx->blk_tot.p, n_blk, (uint32_t *)ctx->misc.p + M_NTOTAL);
    const uint32_t warps_per_block = 8;
    k_gather_intervals<uint2, unsigned long long, IntervalOut><<<(ctx->n_windows + warps_per_block - 1) / warps_per_block, warps_per_block * 32, 0, ctx->s_compute>>>(
        (const unsigned long long *)ctx->rec.p, (const uint2 *)ctx->win_tab.p, (const uint32_t *)ctx->win_out.p,
        (const uint32_t *)ctx->blk_tot.p, ctx->n_windows, (IntervalOut *)ctx->intervals.p, (const uint32_t *)ctx->misc.p + M_ERR);
    k_fill_ends<<<std::max(1, ctx->n_sm * 4), 256, 0, ctx->s_compute>>>((IntervalOut *)ctx->intervals.p,
                                                                       (const uint32_t *)ctx->misc.p + M_NTOTAL, ctx->region_end,
                                                                       (const uint32_t *)ctx->misc.p + M_ERR);
    k_pack_stats<<<1, 32, 0, ctx->s_compute>>>((const unsigned long long *)ctx->stats_padded.p, (unsigned long long *)ctx->counters.p);
    ctx->launches += 5;
    if (ctx->dh_n) {
        const uint32_t n2 = 2 * ctx->dh_n;
        k_fold_depth_hist<<<(n2 + 255) / 256, 256, 0, ctx->s_compute>>>((const unsigned long long *)ctx->dhist.p, n2,
                                                                     (unsigned long long *)ctx->counters.p + N_STATS + 3 * (size_t)ctx->n_bins);
        ctx->launches += 1;
    }
    if (ctx->runs) {
        // the depth runs through the same scan and gather (win_out / blk_tot are free again: the interval gather is done)
        k_scan_windows_local<uint4><<<n_blk, 1024, 0, ctx->s_compute>>>((const uint4 *)ctx->run_win_tab.p, ctx->n_windows, (uint32_t *)ctx->win_out.p,
                                                                       (uint32_t *)ctx->blk_tot.p, (const uint32_t *)ctx->misc.p + M_ERR);
        k_scan_blocks<<<1, 1024, 0, ctx->s_compute>>>((uint32_t *)ctx->blk_tot.p, n_blk, (uint32_t *)ctx->misc.p + M_RUN_NTOTAL);
        k_gather_intervals<uint4, uint2, uint2><<<(ctx->n_windows + warps_per_block - 1) / warps_per_block, warps_per_block * 32, 0, ctx->s_compute>>>(
            (const uint2 *)ctx->run_rec.p, (const uint4 *)ctx->run_win_tab.p, (const uint32_t *)ctx->win_out.p,
            (const uint32_t *)ctx->blk_tot.p, ctx->n_windows, (uint2 *)ctx->runs_out.p, (const uint32_t *)ctx->misc.p + M_ERR);
        ctx->launches += 3;
    }
    CU(cudaGetLastError());
    return CLB_OK;
}

int alloc_outputs(clb_ctx *ctx) {
    int rc;
    const size_t nw = std::max<size_t>(ctx->n_windows, 1);
    if ((rc = ensure(ctx, ctx->win_tab, nw * sizeof(uint2), false, ctx->s_compute))) return rc;
    if ((rc = ensure(ctx, ctx->win_rec, nw * 3 * sizeof(uint4), false, ctx->s_compute))) return rc;
    if ((rc = ensure(ctx, ctx->win_out, nw * 4, false, ctx->s_compute))) return rc;
    if ((rc = ensure(ctx, ctx->deep_list, nw * 4, false, ctx->s_compute))) return rc;
    if ((rc = ensure(ctx, ctx->gen_list, nw * 4, false, ctx->s_compute))) return rc;
    if ((rc = ensure(ctx, ctx->blk_tot, ((nw + 1023) / 1024 + 1) * 4, false, ctx->s_compute))) return rc;
    if ((rc = ensure(ctx, ctx->rec, (size_t)ctx->rec_cap * 8, false, ctx->s_compute))) return rc;
    if ((rc = ensure(ctx, ctx->intervals, (size_t)ctx->rec_cap * sizeof(IntervalOut), false, ctx->s_compute))) return rc;
    if (ctx->runs) {
        // a position starts at most one run: the region length bounds the records and the runs, so they never overflow
        const size_t rlen = ctx->region_end - ctx->region_start;
        if ((rc = ensure(ctx, ctx->run_win_tab, nw * sizeof(uint4), false, ctx->s_compute))) return rc;
        if ((rc = ensure(ctx, ctx->run_rec, rlen * sizeof(uint2), false, ctx->s_compute))) return rc;
        if ((rc = ensure(ctx, ctx->runs_out, rlen * sizeof(uint2), false, ctx->s_compute))) return rc;
    }
    return CLB_OK;
}

// copy counters + interval count, validate device error bits, then copy the intervals
int fetch_result(clb_ctx *ctx, clb_contig_result *out) {
    const size_t n_cnt = n_counters(ctx);
    const size_t n_misc = ctx->runs ? M_WORDS_RUNS : M_WORDS;
    ctx->dh_fetched = 0; ctx->tl_fetched = 0; ctx->runs_fetched = false;
    ctx->h_counters.resize(n_cnt);
    CU(cudaMemcpyAsync(ctx->h_misc, ctx->misc.p, n_misc * 4, cudaMemcpyDeviceToHost, ctx->s_compute));
    CU(cudaMemcpyAsync(ctx->h_counters.data(), ctx->counters.p, n_cnt * 8, cudaMemcpyDeviceToHost, ctx->s_compute));
    CU(cudaStreamSynchronize(ctx->s_compute));
    const uint32_t e = ctx->h_misc[M_ERR];
    if (e & ERR_UNSORTED) return fail(ctx, CLB_E_INPUT, "read columns are not coordinate sorted (or pos < 0)");
    if (e & ERR_OFFSETS) return fail(ctx, CLB_E_INPUT, "cigar_off / qual_off are not monotone");
    if (e & ERR_QUAL_SPAN) return fail(ctx, CLB_E_UNSUPPORTED, "a window's candidate reads span more than 4 GiB of qualities");
    if (e & ERR_REC_OVERFLOW) return 1;   // caller grows the record buffer and re-runs
    const uint64_t n_iv = ctx->n_windows ? ctx->h_misc[M_NTOTAL] : 0;
    if (n_iv > ctx->h_intervals_cap) {
        if (ctx->h_intervals) cudaFreeHost(ctx->h_intervals);
        ctx->h_intervals = nullptr;
        ctx->h_intervals_cap = std::max<size_t>(n_iv + n_iv / 4, 1024);
        CU(cudaHostAlloc((void **)&ctx->h_intervals, ctx->h_intervals_cap * sizeof(clb_interval), cudaHostAllocDefault));
    }
    if (n_iv) {
        CU(cudaMemcpyAsync(ctx->h_intervals, ctx->intervals.p, n_iv * sizeof(clb_interval), cudaMemcpyDeviceToHost, ctx->s_compute));
        CU(cudaStreamSynchronize(ctx->s_compute));
    }
    ctx->n_intervals = n_iv;
    const uint64_t n_runs = ctx->runs && ctx->n_windows ? ctx->h_misc[M_RUN_NTOTAL] : 0;
    if (ctx->runs) {
        if (n_runs > ctx->h_runs_cap || !ctx->h_runs) {
            if (ctx->h_runs) cudaFreeHost(ctx->h_runs);
            ctx->h_runs = nullptr;
            ctx->h_runs_cap = std::max<size_t>(n_runs + n_runs / 4, 1024);
            CU(cudaHostAlloc((void **)&ctx->h_runs, ctx->h_runs_cap * sizeof(clb_depth_run), cudaHostAllocDefault));
        }
        if (n_runs) {
            CU(cudaMemcpyAsync(ctx->h_runs, ctx->runs_out.p, n_runs * sizeof(clb_depth_run), cudaMemcpyDeviceToHost, ctx->s_compute));
            CU(cudaStreamSynchronize(ctx->s_compute));
        }
    }
    ctx->n_runs = n_runs;
    ctx->d2h_bytes = n_misc * 4 + n_cnt * 8 + n_iv * sizeof(clb_interval) + n_runs * sizeof(clb_depth_run);
    ctx->h_bins.resize(3 * (size_t)ctx->n_bins);
    for (size_t i = 0; i < ctx->h_bins.size(); i++) ctx->h_bins[i] = (uint32_t)ctx->h_counters[N_STATS + i];
    ctx->dh_fetched = ctx->dh_n;                                             // the histograms stay in h_counters, after the bins
    ctx->tl_fetched = ctx->n_tiles;                                          // ... and the tiles after them
    ctx->runs_fetched = ctx->runs;

    float kms = 0, hms = 0, ums = 0;
    for (auto &ep : ctx->ev_upload) { float t = 0; cudaEventElapsedTime(&t, ep.a, ep.b); ums += t; ctx->ev_pool.push_back(ep); }
    for (auto &ep : ctx->ev_kernel) { float t = 0; cudaEventElapsedTime(&t, ep.a, ep.b); kms += t; ctx->ev_pool.push_back(ep); }
    for (auto &ep : ctx->ev_h2d) { float t = 0; cudaEventElapsedTime(&t, ep.a, ep.b); hms += t; ctx->ev_pool.push_back(ep); }
    ctx->ev_kernel.clear(); ctx->ev_h2d.clear(); ctx->ev_upload.clear();

    if (out) {
        memset(out, 0, sizeof *out);
        for (int s = 0; s < 6; s++) out->state_counts[s] = ctx->h_counters[S_COUNT0 + s];
        out->n_covered_bases = ctx->h_counters[S_COVERED];
        out->summed_coverage = ctx->h_counters[S_SUMCOV];
        out->summed_baseq = ctx->h_counters[S_SUMBQ];
        out->summed_mapq = ctx->h_counters[S_SUMMAPQ];
        out->quality_bases = ctx->h_counters[S_QBASES];
        out->n_intervals = n_iv;
        out->intervals = ctx->h_intervals;
        out->n_bins = ctx->n_bins; out->stride = ctx->stride;
        out->bins = ctx->h_bins.data();
        out->region_start = ctx->region_start; out->region_end = ctx->region_end;
        out->kernel_ms = kms; out->h2d_ms = hms; out->upload_ms = ums;
        out->h2d_bytes = ctx->h2d_bytes; out->d2h_bytes = ctx->d2h_bytes;
        out->gpu_launches = ctx->launches;
        out->general_windows = ctx->h_misc[M_GEN_COUNT];
    }
    return CLB_OK;
}

// all kernels of the resident contig, from scratch (used for re-runs and record-buffer growth)
int run_all_resident(clb_ctx *ctx, float *ms, float *pileup_ms = nullptr, float *fast_ms = nullptr, bool sync = true) {
    int rc;
    EvPair ep, ek, ef;
    if ((rc = get_events(ctx, ep))) return rc;
    if ((rc = get_events(ctx, ek))) return rc;
    if ((rc = get_events(ctx, ef))) return rc;
    CU(cudaEventRecord(ep.a, ctx->s_compute));
    if ((rc = reset_accumulators(ctx))) return rc;
    const bool fast_runs = !(ctx->force_general || ctx->long_mode) && ctx->n_windows;
    if ((rc = launch_windows(ctx, 0, ctx->n_windows, &ek, &ef))) return rc;
    if ((rc = launch_compaction(ctx))) return rc;
    CU(cudaEventRecord(ep.b, ctx->s_compute));
    if (!sync) {                                             // enqueue only: the caller waits (clb_refresh_counters / the next synchronous call)
        ctx->ev_pool.push_back(ep); ctx->ev_pool.push_back(ek); ctx->ev_pool.push_back(ef);
        return CLB_OK;
    }
    CU(cudaStreamSynchronize(ctx->s_compute));
    float t = 0;
    CU(cudaEventElapsedTime(&t, ep.a, ep.b));
    if (ms) *ms = t;
    if (pileup_ms) { *pileup_ms = 0; if (ctx->n_windows) CU(cudaEventElapsedTime(pileup_ms, ek.a, ek.b)); }
    if (fast_ms) { *fast_ms = 0; if (fast_runs) CU(cudaEventElapsedTime(fast_ms, ef.a, ef.b)); }
    ctx->ev_pool.push_back(ep); ctx->ev_pool.push_back(ek); ctx->ev_pool.push_back(ef);
    return CLB_OK;
}

}  // namespace

// =================================================================================================
extern "C" {

int clb_abi_version(void) { return CLB_ABI_VERSION; }

uint32_t clb_window_positions(void) { return (uint32_t)WREAL; }

int clb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

clb_ctx *clb_create(int device, const clb_options *opt, char *err, size_t err_len) {
    auto bail = [&](const char *what, cudaError_t e) -> clb_ctx * {
        if (err && err_len) snprintf(err, err_len, "%s: %s", what, cudaGetErrorString(e));
        return nullptr;
    };
    if (!opt) { if (err && err_len) snprintf(err, err_len, "options are NULL"); return nullptr; }
    cudaError_t e;
    int n = 0;
    if ((e = cudaGetDeviceCount(&n)) != cudaSuccess || n == 0)
        return bail("no CUDA device (this library has no CPU fallback)", e == cudaSuccess ? cudaErrorNoDevice : e);
    if (device < 0 || device >= n) { if (err && err_len) snprintf(err, err_len, "device %d out of range (0..%d)", device, n - 1); return nullptr; }
    if ((e = cudaSetDevice(device)) != cudaSuccess) return bail("cudaSetDevice", e);
    clb_ctx *ctx = new clb_ctx();
    ctx->device = device; ctx->opt = *opt;
    if ((e = cudaStreamCreateWithFlags(&ctx->s_own, cudaStreamNonBlocking)) != cudaSuccess) { delete ctx; return bail("cudaStreamCreate", e); }
    if ((e = cudaStreamCreateWithFlags(&ctx->s_copy, cudaStreamNonBlocking)) != cudaSuccess) { delete ctx; return bail("cudaStreamCreate", e); }
    ctx->s_compute = ctx->s_own;
    cudaEventCreateWithFlags(&ctx->ev_copy, cudaEventDisableTiming);
    {
        const char *fg = getenv("CLB_FORCE_GENERAL");
        ctx->force_general = fg && fg[0] && fg[0] != '0';
    }
    for (int v = 0; v < 32; v++)                             // every instantiation of the pileup kernels
        with_variant(v & 1, v & 2, (unsigned)v >> 2, [&](auto h, auto d, auto x) {
            constexpr bool H = decltype(h)::value, D = decltype(d)::value; constexpr unsigned X = decltype(x)::value;
            const cudaFuncAttribute smem = cudaFuncAttributeMaxDynamicSharedMemorySize;
            if (e == cudaSuccess) e = cudaFuncSetAttribute(k_pileup_general<H, D, X>, smem, (int)SMEM_BYTES);
            if (e == cudaSuccess) e = cudaFuncSetAttribute(k_pileup_classify_deep<H, D, X>, smem, (int)SMEM_BYTES_DEEP);
            if (e == cudaSuccess) e = cudaFuncSetAttribute(k_pileup_fast<H, D, X>, smem, (int)F_SMEM);
        });
    if (e != cudaSuccess) { clb_destroy(ctx); return bail("cudaFuncSetAttribute (pileup kernels)", e); }
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->max_ctas_per_sm, k_pileup_general<false, false>, NT, SMEM_BYTES);
    cudaDeviceGetAttribute(&ctx->n_sm, cudaDevAttrMultiProcessorCount, device);
    if ((e = cudaMalloc((void **)&ctx->d_first_tab, 65536 * 4 + WIN_TABLE_BYTES + 256)) != cudaSuccess) { clb_destroy(ctx); return bail("cudaMalloc", e); }
    k_first_table<<<65536 / 256, 256, 0, ctx->s_compute>>>(ctx->d_first_tab, (uint8_t *)(ctx->d_first_tab + 65536) + WIN_TABLE_BYTES, opt->max_low_mapq_fraction);
    k_window_tables<<<1, 256, 0, ctx->s_compute>>>(ctx->d_first_tab + 65536, opt->max_low_mapq_fraction);
    if ((e = cudaHostAlloc((void **)&ctx->h_misc, M_WORDS_RUNS * 4, cudaHostAllocDefault)) != cudaSuccess) { clb_destroy(ctx); return bail("cudaHostAlloc", e); }
    if ((e = cudaStreamSynchronize(ctx->s_compute)) != cudaSuccess) { clb_destroy(ctx); return bail("first-table kernel", e); }
    return ctx;
}

void clb_destroy(clb_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    for (DevBuf *b : {&ctx->pos, &ctx->flag, &ctx->mapq, &ctx->cigar_off, &ctx->cigar, &ctx->qual_off, &ctx->qual, &ctx->read_end, &ctx->cigar_ckpt,
                      &ctx->nmask, &ctx->ref_ascii, &ctx->stats_padded, &ctx->counters, &ctx->rec, &ctx->win_tab, &ctx->win_rec,
                      &ctx->win_out, &ctx->deep_list, &ctx->intervals, &ctx->misc, &ctx->gen_list, &ctx->blk_tot, &ctx->dhist, &ctx->run_rec, &ctx->run_win_tab, &ctx->runs_out, &ctx->dbg_raw, &ctx->dbg_qc, &ctx->dbg_low, &ctx->dbg_state, &ctx->timing})
        release(*b);
    if (ctx->d_first_tab) cudaFree(ctx->d_first_tab);
    if (ctx->h_intervals) cudaFreeHost(ctx->h_intervals);
    if (ctx->h_runs) cudaFreeHost(ctx->h_runs);
    if (ctx->h_misc) cudaFreeHost(ctx->h_misc);
    for (auto &ep : ctx->ev_pool) { cudaEventDestroy(ep.a); cudaEventDestroy(ep.b); }
    for (auto &ep : ctx->ev_kernel) { cudaEventDestroy(ep.a); cudaEventDestroy(ep.b); }
    for (auto &ep : ctx->ev_h2d) { cudaEventDestroy(ep.a); cudaEventDestroy(ep.b); }
    for (auto &ep : ctx->ev_upload) { cudaEventDestroy(ep.a); cudaEventDestroy(ep.b); }
    if (ctx->ev_copy) cudaEventDestroy(ctx->ev_copy);
    if (ctx->s_own) cudaStreamDestroy(ctx->s_own);
    if (ctx->s_copy) cudaStreamDestroy(ctx->s_copy);
    delete ctx;
}

const char *clb_last_error(const clb_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int clb_set_stream(clb_ctx *ctx, void *cuda_stream) {
    if (!ctx) return CLB_E_INVALID;
    CU(cudaStreamSynchronize(ctx->s_compute));
    ctx->s_compute = cuda_stream ? (cudaStream_t)cuda_stream : ctx->s_own;
    return CLB_OK;
}

int clb_bin_geometry(const char *name, uint32_t contig_len, uint32_t largest_contig_len, uint32_t *stride, uint32_t *n_bins) {
    // histogram_plotter.rs:419-431 (stride) and :75 (array size); callable_profiler.rs:73-77 (chrM uses its own length)
    const bool is_m = name && strcmp(name, "chrM") == 0;
    const uint32_t s = is_m ? (16569u + 200u - 1u) / 200u : (uint32_t)(((uint64_t)largest_contig_len + 2000u - 1u) / 2000u);
    if (stride) *stride = s;
    if (n_bins) *n_bins = s ? contig_len / s + 1 : 0;
    return s ? CLB_OK : CLB_E_INVALID;
}

int clb_begin_contig(clb_ctx *ctx, int32_t tid, const char *name, uint32_t contig_len, const void *ref, uint64_t ref_len,
                     int ref_kind, uint32_t largest_contig_len, uint32_t region_start, uint32_t region_end, uint32_t max_ref_span) {
    if (!ctx) return CLB_E_INVALID;
    if (region_end > contig_len || region_start > region_end) return fail(ctx, CLB_E_INVALID, "bad region [%u,%u) for contig length %u", region_start, region_end, contig_len);
    CU(cudaSetDevice(ctx->device));
    int rc;
    ctx->tid = tid; ctx->name = name ? name : ""; ctx->contig_len = contig_len; ctx->largest = largest_contig_len;
    ctx->region_start = region_start; ctx->region_end = region_end;
    ctx->n_windows = (uint32_t)(((uint64_t)(region_end - region_start) + WREAL - 1) / WREAL);
    ctx->windows_done = 0;
    ctx->n_reads = ctx->n_cigar = ctx->n_qual = 0; ctx->last_pos = -1;
    ctx->long_mode = false; ctx->span_on_device = (max_ref_span == 0);
    ctx->h2d_bytes = 0; ctx->d2h_bytes = 0; ctx->launches = 0; ctx->n_intervals = 0;
    ctx->dbg = false;
    ctx->dh_n = ctx->dh_next; ctx->dh_fetched = 0;
    ctx->tl_len = ctx->tl_next; ctx->tl_fetched = 0;
    ctx->runs = ctx->runs_next; ctx->runs_fetched = false; ctx->n_runs = 0;
    ctx->n_tiles = ctx->tl_len ? (uint32_t)(((uint64_t)contig_len + ctx->tl_len - 1) / ctx->tl_len) : 0u;
    clb_bin_geometry(ctx->name.c_str(), contig_len, largest_contig_len, &ctx->stride, &ctx->n_bins);

    // reference -> bit-packed N mask, padded so every window can read two words past its last entry
    const size_t n_words = ((size_t)contig_len + WN) / 32 + 4;
    if ((rc = ensure(ctx, ctx->nmask, n_words * 4, false, ctx->s_compute))) return rc;
    EvPair ep; if ((rc = get_events(ctx, ep))) return rc;
    CU(cudaEventRecord(ep.a, ctx->s_compute));
    CU(cudaMemsetAsync(ctx->nmask.p, 0, n_words * 4, ctx->s_compute));
    if (ref_kind == 1) {
        if (ref && contig_len) {
            const size_t w = ((size_t)contig_len + 31) / 32;
            CU(cudaMemcpyAsync(ctx->nmask.p, ref, w * 4, cudaMemcpyHostToDevice, ctx->s_compute));
            ctx->h2d_bytes += w * 4;
        }
    } else if (ref_kind == 0) {
        const uint64_t use = ref ? std::min<uint64_t>(ref_len, contig_len) : 0;
        if (use) {
            if ((rc = ensure(ctx, ctx->ref_ascii, use + 64, false, ctx->s_compute))) return rc;
            CU(cudaMemcpyAsync(ctx->ref_ascii.p, ref, use, cudaMemcpyHostToDevice, ctx->s_compute));
            ctx->h2d_bytes += use;
        }
        if (contig_len) {
            const uint32_t nw = (uint32_t)(((uint64_t)contig_len + 31) / 32);
            EvPair eu; if ((rc = get_events(ctx, eu))) return rc;
            CU(cudaEventRecord(eu.a, ctx->s_compute));
            k_nmask_from_ascii<<<(nw + 255) / 256, 256, 0, ctx->s_compute>>>((const uint8_t *)ctx->ref_ascii.p, use, contig_len, (uint32_t *)ctx->nmask.p, nw);
            CU(cudaEventRecord(eu.b, ctx->s_compute));
            ctx->ev_upload.push_back(eu);
            ctx->launches++;
        }
    } else return fail(ctx, CLB_E_INVALID, "ref_kind must be 0 (ASCII) or 1 (N-mask bits)");
    CU(cudaEventRecord(ep.b, ctx->s_compute));
    ctx->ev_h2d.push_back(ep);

    if ((rc = ensure(ctx, ctx->misc, M_WORDS_RUNS * 4, false, ctx->s_compute))) return rc;
    if ((rc = ensure(ctx, ctx->stats_padded, (size_t)N_STATS * STAT_STRIDE * 8, false, ctx->s_compute))) return rc;
    if ((rc = ensure(ctx, ctx->counters, n_counters(ctx) * 8, false, ctx->s_compute))) return rc;
    if (ctx->dh_n && (rc = ensure(ctx, ctx->dhist, (size_t)DH_SLOTS * 2 * ctx->dh_n * 8, false, ctx->s_compute))) return rc;
    const uint64_t rlen = region_end - region_start;
    ctx->rec_cap = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(rlen / 4 + 4096, 1u << 16), (uint64_t)rlen + 16);
    if ((rc = alloc_outputs(ctx))) return rc;
    if ((rc = reset_accumulators(ctx))) return rc;
    CU(cudaMemcpyAsync((uint32_t *)ctx->misc.p + M_MAXSPAN, &max_ref_span, 4, cudaMemcpyHostToDevice, ctx->s_compute));
    CU(cudaMemsetAsync((uint32_t *)ctx->misc.p + M_MAXQLEN, 0, 4, ctx->s_compute));
    // offsets column entry 0
    if ((rc = ensure(ctx, ctx->cigar_off, 4096, false, ctx->s_compute))) return rc;
    if ((rc = ensure(ctx, ctx->qual_off, 4096, false, ctx->s_compute))) return rc;
    CU(cudaMemsetAsync(ctx->cigar_off.p, 0, 4, ctx->s_compute));
    CU(cudaMemsetAsync(ctx->qual_off.p, 0, 8, ctx->s_compute));
    CU(cudaStreamSynchronize(ctx->s_compute));
    ctx->in_contig = true; ctx->finished = false;
    return CLB_OK;
}

int clb_reserve(clb_ctx *ctx, uint64_t n_reads, uint64_t n_cigar, uint64_t n_qual) {
    if (!ctx || !ctx->in_contig) return fail(ctx, CLB_E_INVALID, "clb_reserve outside a contig");
    int rc;
    cudaStream_t s = ctx->s_copy;
    if ((rc = ensure(ctx, ctx->pos, (n_reads + 1) * 4, true, s))) return rc;
    if ((rc = ensure(ctx, ctx->flag, (n_reads + 1) * 2, true, s))) return rc;
    if ((rc = ensure(ctx, ctx->mapq, n_reads + 16, true, s))) return rc;
    if ((rc = ensure(ctx, ctx->cigar_off, (n_reads + 2) * 4, true, s))) return rc;
    if ((rc = ensure(ctx, ctx->qual_off, (n_reads + 2) * 8, true, s))) return rc;
    if ((rc = ensure(ctx, ctx->cigar, (n_cigar + 4) * 4, true, s))) return rc;
    if ((rc = ensure(ctx, ctx->qual, n_qual + 64, true, s))) return rc;
    return CLB_OK;
}

int clb_push_reads(clb_ctx *ctx, const clb_read_batch *b) {
    if (!ctx || !ctx->in_contig || ctx->finished) return fail(ctx, CLB_E_INVALID, "clb_push_reads outside an open contig");
    if (!b) return fail(ctx, CLB_E_INVALID, "batch is NULL");
    if (b->n_reads == 0) return CLB_OK;
    if (ctx->n_reads + b->n_reads >= 0xffffffffull || ctx->n_cigar + b->n_cigar >= 0xffffffffull)
        return fail(ctx, CLB_E_UNSUPPORTED, "more than 2^32 reads or CIGAR ops in one contig");
    if (!b->pos || !b->flag || !b->mapq || !b->cigar_off || !b->qual_off || (b->n_cigar && !b->cigar) || (b->n_qual && !b->qual))
        return fail(ctx, CLB_E_INVALID, "batch has NULL columns");
    if (b->cigar_off[0] != 0 || b->qual_off[0] != 0) return fail(ctx, CLB_E_INPUT, "batch offsets must start at 0");
    if (b->cigar_off[b->n_reads] != b->n_cigar || b->qual_off[b->n_reads] != b->n_qual) return fail(ctx, CLB_E_INPUT, "batch offsets do not end at n_cigar / n_qual");
    if (b->pos[0] < 0 || (long long)b->pos[0] < ctx->last_pos) return fail(ctx, CLB_E_INPUT, "read columns are not coordinate sorted (or pos < 0)");
    CU(cudaSetDevice(ctx->device));
    int rc;
    if ((rc = clb_reserve(ctx, ctx->n_reads + b->n_reads, ctx->n_cigar + b->n_cigar, ctx->n_qual + b->n_qual))) return rc;
    const uint32_t r0 = (uint32_t)ctx->n_reads, n = (uint32_t)b->n_reads;
    cudaStream_t s = ctx->s_copy;
    EvPair ep; if ((rc = get_events(ctx, ep))) return rc;
    CU(cudaEventRecord(ep.a, s));
    CU(cudaMemcpyAsync((int32_t *)ctx->pos.p + r0, b->pos, (size_t)n * 4, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync((uint16_t *)ctx->flag.p + r0, b->flag, (size_t)n * 2, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync((uint8_t *)ctx->mapq.p + r0, b->mapq, (size_t)n, cudaMemcpyHostToDevice, s));
    // entry r0 of the offset columns is the previous batch's end and may be in use: copy entries 1..n only
    CU(cudaMemcpyAsync((uint32_t *)ctx->cigar_off.p + r0 + 1, b->cigar_off + 1, (size_t)n * 4, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync((uint64_t *)ctx->qual_off.p + r0 + 1, b->qual_off + 1, (size_t)n * 8, cudaMemcpyHostToDevice, s));
    if (b->n_cigar) CU(cudaMemcpyAsync((uint32_t *)ctx->cigar.p + ctx->n_cigar, b->cigar, (size_t)b->n_cigar * 4, cudaMemcpyHostToDevice, s));
    if (b->n_qual) CU(cudaMemcpyAsync((uint8_t *)ctx->qual.p + ctx->n_qual, b->qual, (size_t)b->n_qual, cudaMemcpyHostToDevice, s));
    CU(cudaEventRecord(ep.b, s));
    ctx->ev_h2d.push_back(ep);
    ctx->h2d_bytes += (uint64_t)n * (4 + 2 + 1 + 4 + 8) + b->n_cigar * 4 + b->n_qual;

    // compute stream: wait for the copies, validate + rebase, optional read ends / max span
    CU(cudaEventRecord(ctx->ev_copy, s));
    CU(cudaStreamWaitEvent(ctx->s_compute, ctx->ev_copy, 0));
    EvPair ek; if ((rc = get_events(ctx, ek))) return rc;
    EvPair eu; if ((rc = get_events(ctx, eu))) return rc;
    CU(cudaEventRecord(ek.a, ctx->s_compute));
    CU(cudaEventRecord(eu.a, ctx->s_compute));
    const uint32_t nb = (n + 255) / 256;
    k_validate_batch<<<nb, 256, 0, ctx->s_compute>>>((const int32_t *)ctx->pos.p, (const uint32_t *)ctx->cigar_off.p,
                                                     (const uint64_t *)ctx->qual_off.p, r0, n, (uint32_t *)ctx->misc.p + M_ERR,
                                                     (uint32_t *)ctx->misc.p + M_MAXQLEN);
    k_rebase_batch<<<nb, 256, 0, ctx->s_compute>>>((uint32_t *)ctx->cigar_off.p, (uint64_t *)ctx->qual_off.p, r0, n,
                                                   (uint32_t)ctx->n_cigar, ctx->n_qual);
    ctx->launches += 2;
    // Long-read mode (read ends + CIGAR checkpoints, every window on the general kernel) starts with the first batch that
    // looks like long reads -- normally the first batch of the contig; if it is a later one, the reads already resident are
    // checkpointed too (windows launched before the switch stay valid: results do not depend on which kernel took a window).
    uint32_t ck_from = r0;
    if (!ctx->long_mode && b->n_cigar > 4 * b->n_reads) { ctx->long_mode = true; ck_from = 0; }
    if (ctx->long_mode) {
        // read ends, maximum span and CIGAR checkpoints in one pass (one warp per read)
        if ((rc = ensure(ctx, ctx->read_end, ((size_t)r0 + n + 1) * 4, true, ctx->s_compute))) return rc;
        if ((rc = ensure(ctx, ctx->cigar_ckpt, ((ctx->n_cigar + b->n_cigar) / 32 + 2) * sizeof(uint2), true, ctx->s_compute))) return rc;
        k_cigar_checkpoints<<<(r0 + n - ck_from + 7) / 8, 256, 0, ctx->s_compute>>>((const int32_t *)ctx->pos.p, (const uint32_t *)ctx->cigar_off.p,
                                                                     (const uint32_t *)ctx->cigar.p, ck_from, r0 + n, (uint32_t *)ctx->read_end.p,
                                                                     ctx->span_on_device ? (uint32_t *)ctx->misc.p + M_MAXSPAN : nullptr,
                                                                     (uint2 *)ctx->cigar_ckpt.p);
        ctx->launches++;
    } else if (ctx->span_on_device) {
        k_read_end<<<nb, 256, 0, ctx->s_compute>>>((const int32_t *)ctx->pos.p, (const uint32_t *)ctx->cigar_off.p, (const uint32_t *)ctx->cigar.p,
                                                   r0, r0 + n, nullptr, (uint32_t *)ctx->misc.p + M_MAXSPAN);
        ctx->launches++;
    }
    CU(cudaEventRecord(eu.b, ctx->s_compute));                     // upload-time helper kernels of this batch
    ctx->ev_upload.push_back(eu);
    ctx->n_reads += n; ctx->n_cigar += b->n_cigar; ctx->n_qual += b->n_qual;
    ctx->last_pos = b->pos[n - 1];

    // windows whose exclusive end is <= the last position seen can no longer receive reads
    uint32_t ready = 0;
    if (ctx->last_pos > (long long)ctx->region_start)
        ready = (uint32_t)std::min<uint64_t>(ctx->n_windows, (uint64_t)(ctx->last_pos - ctx->region_start) / WREAL);
    if (ready > ctx->windows_done) {
        if ((rc = launch_windows(ctx, ctx->windows_done, ready))) return rc;
        ctx->windows_done = ready;
    }
    CU(cudaEventRecord(ek.b, ctx->s_compute));
    ctx->ev_kernel.push_back(ek);
    CU(cudaGetLastError());
    return CLB_OK;
}

int clb_finish_contig(clb_ctx *ctx, clb_contig_result *out) {
    if (!ctx || !ctx->in_contig) return fail(ctx, CLB_E_INVALID, "clb_finish_contig without clb_begin_contig");
    CU(cudaSetDevice(ctx->device));
    int rc;
    if (!ctx->finished) {
        EvPair ek; if ((rc = get_events(ctx, ek))) return rc;
        CU(cudaEventRecord(ek.a, ctx->s_compute));
        if ((rc = launch_windows(ctx, ctx->windows_done, ctx->n_windows))) return rc;
        ctx->windows_done = ctx->n_windows;
        if ((rc = launch_compaction(ctx))) return rc;
        CU(cudaEventRecord(ek.b, ctx->s_compute));
        ctx->ev_kernel.push_back(ek);
        ctx->finished = true;
    }
    rc = fetch_result(ctx, out);
    while (rc == 1) {       // interval record buffer was too small: grow to the demanded size and re-run
        const uint32_t need = ctx->h_misc[M_CURSOR];
        ctx->rec_cap = (uint32_t)std::min<uint64_t>((uint64_t)need + need / 8 + 1024, (uint64_t)(ctx->region_end - ctx->region_start) + 16);
        if ((rc = alloc_outputs(ctx))) return rc;
        float ms = 0;
        if ((rc = run_all_resident(ctx, &ms))) return rc;
        rc = fetch_result(ctx, out);
        if (out && rc == CLB_OK) out->kernel_ms = ms;
    }
    return rc;
}

int clb_rerun_resident(clb_ctx *ctx, clb_contig_result *out, float *ms) {
    if (!ctx || !ctx->in_contig || !ctx->finished) return fail(ctx, CLB_E_INVALID, "clb_rerun_resident needs a finished contig");
    CU(cudaSetDevice(ctx->device));
    int rc;
    const uint32_t l0 = ctx->launches;
    float t = 0, tp = 0, tf = 0;
    if ((rc = run_all_resident(ctx, &t, &tp, &tf, out != nullptr || ms != nullptr))) return rc;
    if (ms) *ms = t;
    if (out) {
        rc = fetch_result(ctx, out);
        if (rc == 1) return fail(ctx, CLB_E_CUDA, "record buffer overflow on re-run");
        if (rc) return rc;
        out->kernel_ms = t; out->pileup_ms = tp; out->fast_ms = tf;
        out->gpu_launches = ctx->launches - l0;
        out->general_windows = ctx->h_misc[M_GEN_COUNT];
    }
    return CLB_OK;
}

void *clb_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}

void clb_host_free(void *p) { if (p) cudaFreeHost(p); }

int clb_wait_uploads(clb_ctx *ctx) {
    if (!ctx) return CLB_E_INVALID;
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->s_copy));
    return CLB_OK;
}

int clb_counters_device(clb_ctx *ctx, void **dev_ptr, uint64_t *n_u64) {
    if (!ctx || !ctx->in_contig) return fail(ctx, CLB_E_INVALID, "no contig");
    if (dev_ptr) *dev_ptr = ctx->counters.p;
    if (n_u64) *n_u64 = (uint64_t)n_counters(ctx);
    return CLB_OK;
}

int clb_refresh_counters(clb_ctx *ctx, clb_contig_result *out) {
    if (!ctx || !ctx->in_contig || !ctx->finished) return fail(ctx, CLB_E_INVALID, "clb_refresh_counters needs a finished contig");
    CU(cudaSetDevice(ctx->device));
    CU(cudaDeviceSynchronize());     // the reduction may have run on a stream we do not own
    return fetch_result(ctx, out);
}

int clb_set_depth_histogram(clb_ctx *ctx, uint32_t n_bins) {
    if (!ctx) return CLB_E_INVALID;
    if (ctx->in_contig && !ctx->finished) return fail(ctx, CLB_E_INVALID, "clb_set_depth_histogram while a contig is open");
    if (n_bins != 0 && (n_bins < 2 || n_bins > 65536)) return fail(ctx, CLB_E_INVALID, "depth histogram bins %u: 0 (off) or 2..65536", n_bins);
    ctx->dh_next = n_bins;
    return CLB_OK;
}

int clb_depth_histogram(const clb_ctx *ctx, const uint64_t **raw, const uint64_t **qc, uint32_t *n_bins) {
    if (!ctx) return CLB_E_INVALID;
    const uint32_t n = ctx->dh_fetched;
    const unsigned long long *h = n ? ctx->h_counters.data() + N_STATS + 3 * (size_t)ctx->n_bins : nullptr;
    if (raw) *raw = (const uint64_t *)h;
    if (qc) *qc = n ? (const uint64_t *)(h + n) : nullptr;
    if (n_bins) *n_bins = n;
    return CLB_OK;
}

int clb_set_depth_tiles(clb_ctx *ctx, uint32_t tile_len) {
    if (!ctx) return CLB_E_INVALID;
    if (ctx->in_contig && !ctx->finished) return fail(ctx, CLB_E_INVALID, "clb_set_depth_tiles while a contig is open");
    if (tile_len != 0 && (tile_len < 256 || tile_len > 0x80000000u)) return fail(ctx, CLB_E_INVALID, "depth tile length %u: 0 (off) or 256..2^31", tile_len);
    ctx->tl_next = tile_len;
    return CLB_OK;
}

int clb_depth_tiles(const clb_ctx *ctx, const uint64_t **territory, const uint64_t **callable, const uint64_t **raw_sum,
                    const uint64_t **qc_sum, uint32_t *n_tiles, uint32_t *tile_len) {
    if (!ctx) return CLB_E_INVALID;
    const uint32_t n = ctx->tl_fetched;
    const uint64_t *t = n ? (const uint64_t *)ctx->h_counters.data() + tiles_offset(ctx) : nullptr;
    if (territory) *territory = t;
    if (callable) *callable = n ? t + n : nullptr;
    if (raw_sum) *raw_sum = n ? t + 2 * (size_t)n : nullptr;
    if (qc_sum) *qc_sum = n ? t + 3 * (size_t)n : nullptr;
    if (n_tiles) *n_tiles = n;
    if (tile_len) *tile_len = n ? ctx->tl_len : 0u;
    return CLB_OK;
}

int clb_set_depth_runs(clb_ctx *ctx, int on) {
    if (!ctx) return CLB_E_INVALID;
    if (ctx->in_contig && !ctx->finished) return fail(ctx, CLB_E_INVALID, "clb_set_depth_runs while a contig is open");
    ctx->runs_next = on != 0;
    return CLB_OK;
}

int clb_depth_runs(const clb_ctx *ctx, const clb_depth_run **runs, uint64_t *n_runs) {
    if (!ctx) return CLB_E_INVALID;
    if (runs) *runs = ctx->runs_fetched ? ctx->h_runs : nullptr;
    if (n_runs) *n_runs = ctx->runs_fetched ? ctx->n_runs : 0;
    return CLB_OK;
}

static void *g_nccl_allreduce = nullptr;

int clb_set_nccl_allreduce(void *nccl_allreduce_fn) { g_nccl_allreduce = nccl_allreduce_fn; return CLB_OK; }

int clb_allreduce_nccl(clb_ctx *ctx, void *nccl_comm) {
    if (!ctx || !ctx->in_contig || !ctx->finished) return fail(ctx, CLB_E_INVALID, "clb_allreduce_nccl needs a finished contig");
    if (!nccl_comm) return fail(ctx, CLB_E_INVALID, "nccl_comm is NULL");
    // ncclAllReduce of the NCCL build that owns the communicator: the one the host registered, else the first one visible
    // in this process, else libnccl.so.2
    typedef int (*allreduce_fn)(const void *, void *, size_t, int, int, void *, cudaStream_t);
    allreduce_fn fn = (allreduce_fn)g_nccl_allreduce;
    if (!fn) {
        fn = (allreduce_fn)dlsym(RTLD_DEFAULT, "ncclAllReduce");
        if (!fn) { void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL); if (h) fn = (allreduce_fn)dlsym(h, "ncclAllReduce"); }
        if (!fn) return fail(ctx, CLB_E_UNSUPPORTED, "ncclAllReduce not found in this process");
    }
    CU(cudaSetDevice(ctx->device));
    const size_t n = n_counters(ctx);
    const int ncclUint64 = 5, ncclSum = 0;       // nccl.h: ncclDataType_t / ncclRedOp_t (stable since NCCL 2.0)
    const int r = fn(ctx->counters.p, ctx->counters.p, n, ncclUint64, ncclSum, nccl_comm, ctx->s_compute);
    if (r != 0) return fail(ctx, CLB_E_CUDA, "ncclAllReduce returned %d", r);
    return CLB_OK;                               // asynchronous on the compute stream, like the kernels
}

/* developer hook (not part of the public header): per-window clock64 stamps of the next runs; needs a library
 * built with -DCLB_PHASE_TIMING (the stamps are compiled out of production builds) */
int clb_debug_timing(clb_ctx *ctx, long long *out, uint32_t max_windows, uint32_t *n_windows) {
#ifndef CLB_PHASE_TIMING
    (void)out; (void)max_windows; (void)n_windows;
    return fail(ctx, CLB_E_UNSUPPORTED, "library built without -DCLB_PHASE_TIMING");
#else
    if (!ctx || !ctx->in_contig || !ctx->finished) return CLB_E_INVALID;
    int rc;
    const size_t n = std::min<size_t>(ctx->n_windows, max_windows);
    if ((rc = ensure(ctx, ctx->timing, (size_t)ctx->n_windows * 64, false, ctx->s_compute))) return rc;
    rc = run_all_resident(ctx, nullptr);
    if (rc) return rc;
    CU(cudaMemcpy(out, ctx->timing.p, n * 64, cudaMemcpyDeviceToHost));
    if (n_windows) *n_windows = (uint32_t)n;
    release(ctx->timing);
    return CLB_OK;
#endif
}

/* developer hook (not part of the public header): number of out-of-bounds accesses the kernels of a -DCLB_BOUNDS_CHECK
 * build caught (and skipped) since the last call; always 0 in production builds */
int clb_debug_bounds(clb_ctx *ctx, uint32_t *violations, int *checked_build) {
    if (!ctx) return CLB_E_INVALID;
    CU(cudaSetDevice(ctx->device));
    CU(cudaDeviceSynchronize());
    unsigned int v = 0, zero = 0;
    CU(cudaMemcpyFromSymbol(&v, g_clb_bounds_violations, sizeof v));
    CU(cudaMemcpyToSymbol(g_clb_bounds_violations, &zero, sizeof zero));
    if (violations) *violations = v;
#ifdef CLB_BOUNDS_CHECK
    if (checked_build) *checked_build = 1;
#else
    if (checked_build) *checked_build = 0;
#endif
    return CLB_OK;
}

int clb_debug_per_base(clb_ctx *ctx, uint32_t *raw, uint32_t *qc, uint32_t *low, uint8_t *state) {
    if (!ctx || !ctx->in_contig || !ctx->finished) return fail(ctx, CLB_E_INVALID, "clb_debug_per_base needs a finished contig");
    CU(cudaSetDevice(ctx->device));
    int rc;
    const size_t n = ctx->region_end - ctx->region_start;
    if (n == 0) return CLB_OK;
    if ((rc = ensure(ctx, ctx->dbg_raw, n * 4, false, ctx->s_compute))) return rc;
    if ((rc = ensure(ctx, ctx->dbg_qc, n * 4, false, ctx->s_compute))) return rc;
    if ((rc = ensure(ctx, ctx->dbg_low, n * 4, false, ctx->s_compute))) return rc;
    if ((rc = ensure(ctx, ctx->dbg_state, n, false, ctx->s_compute))) return rc;
    ctx->dbg = true;
    rc = run_all_resident(ctx, nullptr);
    ctx->dbg = false;
    if (rc) return rc;
    if (raw) CU(cudaMemcpy(raw, ctx->dbg_raw.p, n * 4, cudaMemcpyDeviceToHost));
    if (qc) CU(cudaMemcpy(qc, ctx->dbg_qc.p, n * 4, cudaMemcpyDeviceToHost));
    if (low) CU(cudaMemcpy(low, ctx->dbg_low.p, n * 4, cudaMemcpyDeviceToHost));
    if (state) CU(cudaMemcpy(state, ctx->dbg_state.p, n, cudaMemcpyDeviceToHost));
    return CLB_OK;
}

}  // extern "C"
