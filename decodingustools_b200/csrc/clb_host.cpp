// clb_host.cpp -- host half of include/callable_loci_b200.h (no GPU needed).
//
//   clb_admit_reads        htslib bam_plp_push admission as configured by /root/reference/src/callable_loci/mod.rs:55-60
//   clb_bed_writer_*       CallableProfiler::write_state / finish_contig incl. the cross-contig quirks,
//                          /root/reference/src/callable_loci/profilers/callable_profiler.rs:39-87,122-155
//   clb_stitch_intervals   region-shard stitching (multi-GPU, SURVEY.md section 8(e))
//   clb_bedgraph_writer_*  depth runs as bedGraph text (not in the reference)
#include "../../include/callable_loci_b200.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <functional>
#include <memory>
#include <string>
#include <thread>
#include <vector>

#include <unistd.h>

#include <sched.h>
// host threads this process may use: the cores of its affinity mask (a rank bound to its GPU's cores gets its share,
// not the whole machine), capped at 16
static uint32_t clb_host_threads() {
    cpu_set_t set;
    CPU_ZERO(&set);
    unsigned n = 0;
    if (sched_getaffinity(0, sizeof set, &set) == 0) n = (unsigned)CPU_COUNT(&set);
    if (n == 0) n = std::thread::hardware_concurrency();
    return std::max(1u, std::min(16u, n));
}


static const char *kStateName[6] = {"REF_N", "CALLABLE", "NO_COVERAGE", "LOW_COVERAGE", "EXCESSIVE_COVERAGE", "POOR_MAPPING_QUALITY"};

namespace {

inline uint32_t ref_span(const uint32_t *cigar_off, const uint32_t *cigar, uint64_t i) {
    uint32_t span = 0;
    for (uint32_t c = cigar_off[i]; c < cigar_off[i + 1]; c++) {
        const uint32_t op = cigar[c] & 15u;
        if ((0x18du >> op) & 1u) span += cigar[c] >> 4;                       // M, D, N, =, X
    }
    return span;
}

// The iterator mechanics in closed form (SURVEY.md Appendix A): a record is dropped iff it is not the first record seen
// at its start position and the number of live nodes (admitted records whose end >= pos) has reached maxcnt.  The
// iterator starts at (tid 0, pos 0), so the very first record of tid 0 at pos 0 counts as "not first".  A zero-span
// record that is not first is never retained.  Live nodes are counted in a ring of end positions (O(1) per record,
// O(contig length) in total) instead of a heap.
struct LiveRing {
    std::vector<uint32_t> cnt;      // cnt[e & mask] = live nodes ending at e, for e in [low, low + size)
    uint64_t mask = 0;
    long long low = 0;              // every end < low has expired
    uint64_t live = 0;
    std::vector<long long> far;     // ends beyond the ring (spans longer than expected): min-heap
    void init(uint64_t max_span) {
        uint64_t sz = 1024;
        while (sz < max_span + 2) sz <<= 1;
        cnt.assign(sz, 0); mask = sz - 1; low = 0; live = 0; far.clear();
    }
    void expire_below(long long p) {                       // drop nodes with end < p
        if (p > low) {
            if (live > far.size()) {
                const long long stop = std::min<long long>(p, low + (long long)cnt.size());
                for (long long e = low; e < stop; e++) { uint32_t &c = cnt[(uint64_t)e & mask]; live -= c; c = 0; }
            }
            low = p;
        }
        while (!far.empty() && far.front() < p) { std::pop_heap(far.begin(), far.end(), std::greater<long long>()); far.pop_back(); live--; }
    }
    void add(long long end) {
        if (end < low + (long long)cnt.size()) cnt[(uint64_t)end & mask]++;
        else { far.push_back(end); std::push_heap(far.begin(), far.end(), std::greater<long long>()); }
        live++;
    }
};

// sequential recurrence over records [lo, hi); state = ring + (any, last_pos)
int admit_range(uint32_t maxcnt, uint64_t lo, uint64_t hi, const int32_t *pos, const uint16_t *flag, const uint32_t *cigar_off,
                const uint32_t *cigar, uint8_t *keep, LiveRing &ring, bool &any, long long &last_pos, bool tid0, long long prev) {
    for (uint64_t i = lo; i < hi; i++) {
        keep[i] = 0;
        if (flag[i] & 0x4) continue;
        const long long p = pos[i];
        if (p < prev) return CLB_E_INPUT;
        prev = p;
        const long long end = p + (long long)ref_span(cigar_off, cigar, i);
        const bool same = any ? (p == last_pos) : (tid0 && p == 0);
        any = true;
        ring.expire_below(p);
        if (same) {
            if (ring.live >= (uint64_t)maxcnt) continue;
            if (end > p) { ring.add(end); keep[i] = 1; }
        } else {
            ring.add(end); keep[i] = 1;
        }
        last_pos = p;
    }
    return CLB_OK;
}

}  // namespace

extern "C" int clb_admit_reads(int32_t tid, uint32_t maxcnt, uint64_t n_reads, const int32_t *pos, const uint16_t *flag,
                               const uint32_t *cigar_off, const uint32_t *cigar, uint8_t *keep) {
    uint64_t max_span = 0;
    for (uint64_t i = 0; i < n_reads; i++) max_span = std::max<uint64_t>(max_span, ref_span(cigar_off, cigar, i));
    LiveRing ring; ring.init(max_span);
    bool any = false; long long last_pos = -1;
    return admit_range(maxcnt, 0, n_reads, pos, flag, cigar_off, cigar, keep, ring, any, last_pos, tid == 0, -1);
}

// Streaming form for a decoder that sees one record at a time (the C++ `coverage` host packs only admitted records).
struct clb_admitter {
    LiveRing ring; bool any = false; long long last_pos = -1, prev = -1; bool tid0 = false; uint32_t maxcnt = 500;
};
extern "C" clb_admitter *clb_admitter_new(int32_t tid, uint32_t maxcnt) {
    clb_admitter *a = new clb_admitter();
    a->ring.init(65534); a->tid0 = tid == 0; a->maxcnt = maxcnt;      // spans beyond the ring go to its overflow heap
    return a;
}
extern "C" void clb_admitter_free(clb_admitter *a) { delete a; }
extern "C" int clb_admitter_push(clb_admitter *a, int32_t pos, uint16_t flag, const uint32_t *cigar, uint32_t n_cigar) {
    if (!a) return CLB_E_INVALID;
    uint8_t keep = 0;
    const uint32_t off[2] = {0, n_cigar};
    const int rc = admit_range(a->maxcnt, 0, 1, &pos, &flag, off, cigar, &keep, a->ring, a->any, a->last_pos, a->tid0, a->prev);
    if (rc) return rc;
    if (!(flag & 0x4)) a->prev = pos;
    return keep;
}

// Same result, in parallel.  The cap can only fire at record i when at least maxcnt records start within max_span
// before it (live <= #{j < i : pos[j] + max_span >= pos[i]}), i.e. when pos[i - maxcnt] + max_span >= pos[i]: every other
// record is admitted whatever happened before it (zero-span rule aside).  Flagged records form runs; a run is
// replayed sequentially from the live set at its start, which consists of unflagged (hence known) records only once
// runs whose look-back windows touch have been merged.  30x data has no flagged record at all; a uniformly deep contig
// is one run and costs what clb_admit_reads costs.
extern "C" int clb_admit_reads_mt(int32_t tid, uint32_t maxcnt, uint64_t n_reads, const int32_t *pos, const uint16_t *flag,
                                  const uint32_t *cigar_off, const uint32_t *cigar, uint32_t max_ref_span, uint32_t n_threads,
                                  uint8_t *keep, uint64_t *n_replayed) {
    if (n_replayed) *n_replayed = 0;
    if (n_reads == 0) return CLB_OK;
    if (maxcnt == 0) { if (n_replayed) *n_replayed = n_reads; return clb_admit_reads(tid, maxcnt, n_reads, pos, flag, cigar_off, cigar, keep); }
    // automatic thread count: all cores (at most 16) but at least 16384 records per thread; an explicit count is
    // honoured down to 64 records per thread
    if (n_threads == 0) n_threads = (uint32_t)std::min<uint64_t>(clb_host_threads(), (n_reads + 16383) / 16384);
    n_threads = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(n_threads, (n_reads + 63) / 64));
    const uint64_t chunk = (n_reads + n_threads - 1) / n_threads;
    auto parallel = [&](auto &&fn) {
        std::vector<std::thread> th;
        for (uint32_t t = 1; t < n_threads; t++) th.emplace_back([&, t] { fn(t, std::min(n_reads, t * chunk), std::min(n_reads, (t + 1) * chunk)); });
        fn(0, 0, std::min(n_reads, chunk));
        for (auto &x : th) x.join();
    };
    const bool dbg_t = getenv("CLB_ADMIT_DEBUG") != nullptr;
    auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t0 = now();
    // pass 0: sortedness and (when the caller does not know it) the maximum reference span
    std::vector<uint64_t> t_span(n_threads, 0);
    std::vector<int> t_bad(n_threads, 0);
    const bool need_span = max_ref_span == 0;
    parallel([&](uint32_t t, uint64_t lo, uint64_t hi) {
        uint64_t ms = 0; int bad = 0;
        for (uint64_t i = lo; i < hi; i++) {
            if (pos[i] < 0 || (i > 0 && pos[i] < pos[i - 1])) bad = 1;
            if (need_span) ms = std::max<uint64_t>(ms, ref_span(cigar_off, cigar, i));
        }
        t_span[t] = ms; t_bad[t] = bad;
    });
    uint64_t max_span = max_ref_span;
    for (uint32_t t = 0; t < n_threads; t++) {
        max_span = std::max(max_span, t_span[t]);
        if (t_bad[t]) { if (n_replayed) *n_replayed = n_reads; return clb_admit_reads(tid, maxcnt, n_reads, pos, flag, cigar_off, cigar, keep); }   // let the sequential pass judge
    }
    const double t1 = now();
    // pass 1: unflagged records are decided on the spot; flagged ones are collected as runs [first, last]
    struct Run { uint64_t first, last; };
    std::vector<std::vector<Run>> t_runs(n_threads);
    parallel([&](uint32_t t, uint64_t lo, uint64_t hi) {
        std::vector<Run> &runs = t_runs[t];
        for (uint64_t i = lo; i < hi; i++) {
            const bool mapped = !(flag[i] & 0x4);
            if (mapped && i >= maxcnt && (long long)pos[i - maxcnt] + (long long)max_span >= (long long)pos[i]) {
                if (!runs.empty() && runs.back().last + 1 == i) runs.back().last = i; else runs.push_back({i, i});
                keep[i] = 0;
                continue;
            }
            uint8_t k = mapped ? 1 : 0;
            // zero reference span?  Almost every record starts with a reference-consuming op: one load settles it.
            bool zero = false;
            if (mapped) {
                const uint32_t c0 = cigar_off[i], c1 = cigar_off[i + 1];
                const uint32_t v0 = c1 > c0 ? cigar[c0] : 0u;
                zero = !(((0x18du >> (v0 & 15u)) & 1u) && (v0 >> 4)) && ref_span(cigar_off, cigar, i) == 0;
            }
            if (zero) {
                // zero-span record: retained only when first at its position (relative to the previous mapped record)
                long long j = (long long)i - 1;
                while (j >= 0 && (flag[j] & 0x4)) j--;
                if (j >= 0 ? pos[j] == pos[i] : (tid == 0 && pos[i] == 0)) k = 0;
            }
            keep[i] = k;
        }
    });
    if (dbg_t) fprintf(stderr, "clb_admit_reads_mt: %u threads, pass0 %.3f s, pass1 %.3f s\n", n_threads, t1 - t0, now() - t1);
    // merge runs whose look-back windows touch: run B depends on run A when a record of A can still be live at B's start
    std::vector<Run> runs;
    for (auto &v : t_runs) for (const Run &r : v) {
        if (!runs.empty() && (runs.back().last + 1 == r.first || (long long)pos[runs.back().last] + (long long)max_span >= (long long)pos[r.first])) runs.back().last = r.last;
        else runs.push_back(r);
    }
    if (runs.empty()) return CLB_OK;
    uint64_t replayed = 0;
    for (const Run &r : runs) replayed += r.last - r.first + 1;
    if (n_replayed) *n_replayed = replayed;
    // pass 2: replay the runs (in parallel over runs)
    std::atomic<size_t> next{0};
    std::atomic<int> rc_all{CLB_OK};
    auto worker = [&] {
        LiveRing ring; ring.init(max_span);
        for (;;) {
            const size_t ri = next.fetch_add(1);
            if (ri >= runs.size()) break;
            const Run &r = runs[ri];
            ring.init(max_span);
            // live set at the run's start: the records before it that can reach pos[first] (all decided in pass 1)
            const long long p0 = pos[r.first];
            uint64_t b = r.first;
            while (b > 0 && (long long)pos[b - 1] + (long long)max_span >= p0) b--;
            ring.low = p0;
            bool any = false; long long last_pos = -1;
            {   // previous mapped record (for the "first at this position" test)
                long long j = (long long)r.first - 1;
                while (j >= 0 && (flag[j] & 0x4)) j--;
                any = j >= 0; last_pos = j >= 0 ? pos[j] : -1;
            }
            for (uint64_t j = b; j < r.first; j++) {
                if (!keep[j]) continue;
                const long long e = (long long)pos[j] + (long long)ref_span(cigar_off, cigar, j);
                if (e >= p0) ring.add(e);
            }
            const int rc = admit_range(maxcnt, r.first, r.last + 1, pos, flag, cigar_off, cigar, keep, ring, any, last_pos, tid == 0, -1);
            if (rc) rc_all = rc;
        }
    };
    {
        const uint32_t nt = (uint32_t)std::min<size_t>(n_threads, runs.size());
        std::vector<std::thread> th;
        for (uint32_t t = 1; t < nt; t++) th.emplace_back(worker);
        worker();
        for (auto &x : th) x.join();
    }
    return rc_all;
}

extern "C" int clb_compact_reads(const clb_read_batch *in, const uint8_t *keep, int32_t *pos, uint16_t *flag, uint8_t *mapq,
                                 uint32_t *cigar_off, uint32_t *cigar, uint64_t *qual_off, uint8_t *qual, clb_read_batch *out) {
    if (!in || !keep || !out) return CLB_E_INVALID;
    uint64_t n = 0, nc = 0, nq = 0;
    cigar_off[0] = 0; qual_off[0] = 0;
    for (uint64_t i = 0; i < in->n_reads; i++) {
        if (!keep[i]) continue;
        const uint32_t c0 = in->cigar_off[i], c1 = in->cigar_off[i + 1];
        const uint64_t q0 = in->qual_off[i], q1 = in->qual_off[i + 1];
        pos[n] = in->pos[i]; flag[n] = in->flag[i]; mapq[n] = in->mapq[i];
        memcpy(cigar + nc, in->cigar + c0, (size_t)(c1 - c0) * 4); nc += c1 - c0;
        memcpy(qual + nq, in->qual + q0, (size_t)(q1 - q0)); nq += q1 - q0;
        n++;
        cigar_off[n] = (uint32_t)nc; qual_off[n] = nq;
    }
    out->n_reads = n; out->n_cigar = nc; out->n_qual = nq;
    out->pos = pos; out->flag = flag; out->mapq = mapq; out->cigar_off = cigar_off; out->cigar = cigar; out->qual_off = qual_off; out->qual = qual;
    return CLB_OK;
}

extern "C" uint64_t clb_stitch_intervals(const clb_interval *const *shards, const uint64_t *n_per_shard, uint32_t n_shards,
                                         clb_interval *out) {
    uint64_t n = 0;
    for (uint32_t s = 0; s < n_shards; s++) {
        for (uint64_t i = 0; i < n_per_shard[s]; i++) {
            clb_interval iv = shards[s][i];
            if (n > 0 && i == 0 && iv.soft_start && out[n - 1].state == iv.state && out[n - 1].end == iv.start) {
                out[n - 1].end = iv.end;                     // same run continues across the shard seam
                continue;
            }
            iv.soft_start = 0;
            out[n++] = iv;
        }
    }
    return n;
}

// Where a text writer's output goes (a stdio file or memory) and the text formatting of large contigs on several threads.
struct TextSink {
    FILE *fp = nullptr;
    std::string mem;
    bool in_memory = false;
    bool io_failed = false;        // the first failed stdio / pwrite call; add_contig and close report it as CLB_E_IO
    std::vector<char> buf;
    struct Part { std::unique_ptr<char[]> p; size_t cap = 0; };
    std::vector<Part> parts;                // per-thread formatting buffers (reused, never zero-filled)
    void put(const char *s, size_t n) {
        if (in_memory) mem.append(s, n);
        else {
            if (buf.size() + n > (1u << 20)) flush();
            buf.insert(buf.end(), s, s + n);
        }
    }
    void flush() {
        if (fp && !buf.empty()) { if (fwrite(buf.data(), 1, buf.size(), fp) != buf.size()) io_failed = true; buf.clear(); }
    }
    bool open(const char *path) {
        if (!path) { in_memory = true; return true; }
        fp = fopen(path, "wb");
        return fp != nullptr;
    }
    int close() {
        if (fp) { flush(); if (fclose(fp) != 0) io_failed = true; }
        return io_failed ? CLB_E_IO : CLB_OK;
    }
    // Items [0, n) as text, in order: format(part, lo, hi) writes the text of items [lo, hi) into part (growing it) and
    // returns its length.  From 65536 items on (the BED text of a 30x human chromosome is ~100 MB) nt threads format one
    // slice each, then the parts are copied / pwritten to their final offsets in parallel (written in order to a pipe).
    template <typename Format>
    void put_items(uint64_t n, const char *what, Format format) {
        const uint32_t nt = n < (1u << 16) ? 1 : clb_host_threads();
        if (parts.size() < nt) parts.resize(nt);
        if (nt == 1) { put(parts[0].p.get(), format(parts[0], (uint64_t)0, n)); return; }
        const bool dbg_t = getenv("CLB_ADMIT_DEBUG") != nullptr;
        auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
        const double t0 = now();
        std::vector<size_t> sizes(nt, 0);
        const uint64_t per = (n + nt - 1) / nt;
        auto run_threads = [&](auto &&fn) {
            std::vector<std::thread> th;
            for (uint32_t t = 1; t < nt; t++) th.emplace_back(fn, t);
            fn(0);
            for (auto &x : th) x.join();
        };
        run_threads([&](uint32_t t) {
            const uint64_t lo = std::min(n, t * per), hi = std::min(n, lo + per);
            sizes[t] = format(parts[t], lo, hi);
        });
        const double t1 = now();
        std::vector<size_t> off(nt + 1, 0);
        for (uint32_t t = 0; t < nt; t++) off[t + 1] = off[t] + sizes[t];
        if (in_memory) {
            const size_t base = mem.size();
            mem.resize(base + off[nt]);
            run_threads([&](uint32_t t) { memcpy(&mem[base + off[t]], parts[t].p.get(), sizes[t]); });
        } else {
            flush();
            if (fflush(fp) != 0) io_failed = true;
            const off_t base = ftello(fp);
            if (base >= 0) {                                     // a seekable file: every part goes straight to its offset
                const int fd = fileno(fp);
                std::atomic<bool> io_err{false};
                run_threads([&](uint32_t t) {
                    size_t done = 0;
                    while (done < sizes[t]) {
                        const ssize_t r = pwrite(fd, parts[t].p.get() + done, sizes[t] - done, base + (off_t)(off[t] + done));
                        if (r <= 0) { io_err = true; break; }
                        done += (size_t)r;
                    }
                });
                if (io_err || fseeko(fp, base + (off_t)off[nt], SEEK_SET) != 0) io_failed = true;
            } else {                                             // a pipe or a terminal: in order
                for (uint32_t t = 0; t < nt; t++)
                    if (fwrite(parts[t].p.get(), 1, sizes[t], fp) != sizes[t]) io_failed = true;
            }
        }
        if (dbg_t) fprintf(stderr, "%s: %u threads, format %.3f s, output %.3f s (%zu bytes)\n", what, nt, t1 - t0, now() - t1, off[nt]);
    }
};

struct clb_bed_writer : TextSink {
    uint32_t largest = 0;
    bool have_pending = false;     // CallableProfiler::current_state survives finish_contig (quirk Q1)
    std::string pend_name;
    clb_interval pend{};
};

static const uint8_t kStateLen[6] = {5, 8, 11, 12, 18, 20};
// decimal text of v, two digits per step
static inline char *put_u32_fast(char *p, uint32_t v) {
    static const char D[201] =
        "0001020304050607080910111213141516171819202122232425262728293031323334353637383940414243444546474849"
        "5051525354555657585960616263646566676869707172737475767778798081828384858687888990919293949596979899";
    const int nd = v < 10u ? 1 : v < 100u ? 2 : v < 1000u ? 3 : v < 10000u ? 4 : v < 100000u ? 5 : v < 1000000u ? 6 : v < 10000000u ? 7 : v < 100000000u ? 8 : v < 1000000000u ? 9 : 10;
    char *e = p + nd, *q = e;
    while (v >= 100u) { const uint32_t r = v % 100u; v /= 100u; q -= 2; q[0] = D[2 * r]; q[1] = D[2 * r + 1]; }
    if (v >= 10u) { q -= 2; q[0] = D[2 * v]; q[1] = D[2 * v + 1]; } else { *--q = (char)('0' + v); }
    return e;
}

static inline bool binned_state(uint8_t s) { return s == CLB_CALLABLE || s == CLB_POOR_MAPPING_QUALITY || s == CLB_REF_N; }

// The BED lines of iv[lo, hi) (states already validated) into out; returns their length.  *binned |= whether one of them
// has a binned state.
static size_t format_lines(TextSink::Part &out, const std::string &name, const clb_interval *iv, uint64_t lo, uint64_t hi, bool *binned) {
    const size_t max_line = name.size() + 1 + 10 + 1 + 10 + 1 + 20 + 1;
    if (out.cap < (size_t)(hi - lo) * max_line) { out.cap = (size_t)(hi - lo) * max_line; out.p.reset(new char[out.cap]); }
    char *p = out.p.get();
    bool any = false;
    for (uint64_t i = lo; i < hi; i++) {
        memcpy(p, name.data(), name.size()); p += name.size();
        *p++ = '\t'; p = put_u32_fast(p, iv[i].start); *p++ = '\t'; p = put_u32_fast(p, iv[i].end); *p++ = '\t';
        const uint8_t st = iv[i].state;
        memcpy(p, kStateName[st], kStateLen[st]); p += kStateLen[st]; *p++ = '\n';
        any |= binned_state(st);
    }
    *binned |= any;
    return (size_t)(p - out.p.get());
}

extern "C" clb_bed_writer *clb_bed_writer_open(const char *path, uint32_t largest_contig_len) {
    clb_bed_writer *w = new clb_bed_writer();
    w->largest = largest_contig_len;
    if (!w->open(path)) { delete w; return nullptr; }         // File::create truncates: callable_profiler.rs:31
    return w;
}

extern "C" int clb_bed_writer_add_contig(clb_bed_writer *w, const char *name, uint32_t contig_len, const clb_interval *iv, uint64_t n_iv,
                                         uint32_t *bins_inout, uint32_t n_bins, uint32_t stride, int *has_bins) {
    if (!w || !name) return CLB_E_INVALID;
    // intervals must tile [0, contig_len)
    uint32_t expect = 0;
    for (uint64_t i = 0; i < n_iv; i++) {
        if (iv[i].start != expect || iv[i].end <= iv[i].start || iv[i].state > 5) return CLB_E_INPUT;
        if (i > 0 && iv[i].state == iv[i - 1].state) return CLB_E_INPUT;
        expect = iv[i].end;
    }
    if (expect != contig_len) return CLB_E_INPUT;
    const std::string nm(name);
    bool any_range = false;
    if (w->parts.empty()) w->parts.resize(1);
    // Q1: the first position of a contig (or finish_contig of an empty one) flushes the previous contig's
    // last run once more; Q2: that flush also pushes it into THIS contig's coverage_ranges.
    if (w->have_pending) {
        bool binned = false;
        w->put(w->parts[0].p.get(), format_lines(w->parts[0], w->pend_name, &w->pend, 0, 1, &binned));
        if (binned) {
            any_range = true;
            if (bins_inout && n_bins && stride) {
                uint32_t *row = bins_inout + (size_t)(w->pend.state == CLB_CALLABLE ? 0 : w->pend.state == CLB_POOR_MAPPING_QUALITY ? 1 : 2) * n_bins;
                // positions p in [start,end) with p / stride < n_bins  (histogram_plotter.rs:82-98)
                const uint64_t lim = (uint64_t)n_bins * stride;
                const uint64_t a = w->pend.start, b = std::min<uint64_t>(w->pend.end, lim);
                for (uint64_t p = a; p < b;) {
                    const uint64_t bi = p / stride, nxt = std::min<uint64_t>(b, (bi + 1) * stride);
                    row[bi] += (uint32_t)(nxt - p);
                    p = nxt;
                }
            }
        }
    }
    std::atomic<bool> binned{false};
    w->put_items(n_iv, "clb_bed_writer_add_contig", [&](TextSink::Part &part, uint64_t lo, uint64_t hi) {
        bool b = false;
        const size_t len = format_lines(part, nm, iv, lo, hi, &b);
        if (b) binned = true;
        return len;
    });
    if (binned) any_range = true;
    if (n_iv) { w->have_pending = true; w->pend_name = nm; w->pend = iv[n_iv - 1]; }
    if (has_bins) *has_bins = any_range ? 1 : 0;
    return w->io_failed ? CLB_E_IO : CLB_OK;
}

extern "C" const char *clb_bed_writer_buffer(clb_bed_writer *w, uint64_t *len) {
    if (!w) return nullptr;
    if (len) *len = w->mem.size();
    return w->mem.data();
}

extern "C" int clb_bed_writer_close(clb_bed_writer *w) {
    if (!w) return CLB_E_INVALID;
    const int rc = w->close();
    delete w;
    return rc;
}

struct clb_bedgraph_writer : TextSink {};

// The bedGraph lines of runs[lo, hi) (runs[hi] or contig_len ends run hi - 1) into out; returns their length.
static size_t format_runs(TextSink::Part &out, const std::string &name, uint32_t contig_len, const clb_depth_run *runs, uint64_t n,
                          uint64_t lo, uint64_t hi) {
    const size_t max_line = name.size() + 1 + 10 + 1 + 10 + 1 + 10 + 1;
    if (out.cap < (size_t)(hi - lo) * max_line) { out.cap = (size_t)(hi - lo) * max_line; out.p.reset(new char[out.cap]); }
    char *p = out.p.get();
    for (uint64_t i = lo; i < hi; i++) {
        memcpy(p, name.data(), name.size()); p += name.size();
        *p++ = '\t'; p = put_u32_fast(p, runs[i].start); *p++ = '\t'; p = put_u32_fast(p, i + 1 < n ? runs[i + 1].start : contig_len);
        *p++ = '\t'; p = put_u32_fast(p, runs[i].depth); *p++ = '\n';
    }
    return (size_t)(p - out.p.get());
}

extern "C" clb_bedgraph_writer *clb_bedgraph_writer_open(const char *path) {
    clb_bedgraph_writer *w = new clb_bedgraph_writer();
    if (!w->open(path)) { delete w; return nullptr; }
    return w;
}

extern "C" int clb_bedgraph_writer_add_contig(clb_bedgraph_writer *w, const char *name, uint32_t contig_len, const clb_depth_run *runs,
                                              uint64_t n) {
    if (!w || !name || (n && !runs)) return CLB_E_INVALID;
    // runs must tile [0, contig_len): the first starts at 0, starts ascend strictly, the last starts before contig_len
    if ((n == 0) != (contig_len == 0)) return CLB_E_INVALID;
    for (uint64_t i = 0; i < n; i++) {
        if (i == 0 ? runs[0].start != 0 : runs[i].start <= runs[i - 1].start) return CLB_E_INVALID;
    }
    if (n && runs[n - 1].start >= contig_len) return CLB_E_INVALID;
    const std::string nm(name);
    w->put_items(n, "clb_bedgraph_writer_add_contig", [&](TextSink::Part &part, uint64_t lo, uint64_t hi) {
        return format_runs(part, nm, contig_len, runs, n, lo, hi);
    });
    return w->io_failed ? CLB_E_IO : CLB_OK;
}

extern "C" const char *clb_bedgraph_writer_buffer(clb_bedgraph_writer *w, uint64_t *len) {
    if (!w) return nullptr;
    if (len) *len = w->mem.size();
    return w->mem.data();
}

extern "C" int clb_bedgraph_writer_close(clb_bedgraph_writer *w) {
    if (!w) return CLB_E_INVALID;
    const int rc = w->close();
    delete w;
    return rc;
}
