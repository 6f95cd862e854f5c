// coverage_cli.cpp -- `decodingus-tools-b200 coverage`: the reference's `coverage` command on the B200 path.
//
// Host side of the drop-in (SURVEY.md section 8(f), rows N1-N4), written in C++ because this image has no
// Rust toolchain; it only talks to the device through the C ABI of include/callable_loci_b200.h, exactly as a Rust
// host would.  Mirrors, with citations into /root/reference:
//   flags and defaults                     src/cli.rs:14-61
//   run_analysis / contig selection        src/api/coverage.rs:53-115,149-236 (ascending tid, largest non-chrM length)
//   process_single_contig                  src/callable_loci/mod.rs:44-147 (per-base loop replaced by the device)
//   build_coverage_export / natural order  src/callable_loci/report.rs:15-134,337-393
//   get_quality_stats                      src/callable_loci/profilers/contig_profiler.rs:123-158
//   summary.json (written in the CWD)      src/main.rs:67-69, src/export/formats/coverage.rs (field order)
//   detect_aligner / reference build       src/callable_loci/mod.rs:149-177, src/types.rs:100-147
//   BamStats sampler, platform inference, SVG plots, HTML report: report_writer.hpp (citations there)
// What rust-htslib did (BGZF inflate, BAM record decode, faidx) is done in bam_reader.hpp: multi-threaded zlib inflate of BGZF
// blocks, a record scan (sequential, or per selected contig through the .bai when there is one) and an in-memory FASTA contig load.
// The HTML page is wrapped in this tool's own header/footer unless --report-templates points at a reference checkout's
// src/callable_loci/templates (then the page is what the reference writes, byte for byte).
#include "../../../include/callable_loci_b200.h"
#include "bam_reader.hpp"
#include "report_writer.hpp"

#include <algorithm>
#include <atomic>
#include <charconv>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <mutex>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <map>
#include <memory>
#include <set>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

namespace {

[[noreturn]] void die(const std::string &m) { throw std::runtime_error(m); }
using namespace bamio;

inline uint64_t ticks() {
#if defined(__x86_64__)
    return __builtin_ia32_rdtsc();
#else
    return (uint64_t)std::chrono::steady_clock::now().time_since_epoch().count();
#endif
}

// ------------------------------------------------------------------------------------------------ report
struct ContigStats {            // ContigProfiler + CallableProfiler::contig_counts
    std::string name; uint64_t length = 0;
    uint64_t counts[6] = {0, 0, 0, 0, 0, 0};
    uint64_t n_covered = 0, sum_cov = 0, sum_bq = 0, sum_mapq = 0, qbases = 0, n_reads = 0;
};

size_t split_pos(const std::string &s) {
    for (size_t i = 0; i < s.size(); i++) if (isdigit((unsigned char)s[i]) || s[i] == 'X' || s[i] == 'Y' || s[i] == 'M') return i;
    return s.size();
}
void order_key(const std::string &suf, unsigned &cat, uint32_t &num) {
    const char *p = suf.c_str(); if (*p == '+') p++;
    bool ok = *p != 0; uint64_t v = 0;
    for (const char *q = p; *q; q++) { if (*q < '0' || *q > '9') { ok = false; break; } v = v * 10 + (uint64_t)(*q - '0'); if (v > 0xffffffffull) { ok = false; break; } }
    num = 0;
    if (ok) { cat = 0; num = (uint32_t)v; return; }
    cat = suf == "X" ? 1 : suf == "Y" ? 2 : (suf == "M" || suf == "MT") ? 3 : 4;
}
bool contig_less(const std::string &a, const std::string &b) {     // report.rs:339-383
    const size_t sa = split_pos(a), sb = split_pos(b);
    const std::string pa = a.substr(0, sa), pb = b.substr(0, sb);
    if (pa != pb) return pa < pb;
    unsigned ca, cb; uint32_t na, nb;
    order_key(a.substr(sa), ca, na); order_key(b.substr(sb), cb, nb);
    if (ca != cb) return ca < cb;
    if (ca == 0) return na < nb;
    return a.substr(sa) < b.substr(sb);
}

using report::fmt_f64;
using report::jstr;

std::string detect_aligner(const std::string &header_text) {       // callable_loci/mod.rs:149-177
    std::string h = header_text; for (auto &c : h) c = (char)tolower((unsigned char)c);
    auto has = [&](const char *s) { return h.find(s) != std::string::npos; };
    if (has("@pg\tid:bwa-mem2")) return "BWA-MEM2";
    if (has("@pg\tid:bwa")) return "BWA";
    if (has("@pg\tid:minimap2")) return "minimap2";
    if (has("@pg\tid:pbmm2")) return "pbmm2";
    if (has("@pg\tid:bowtie2")) return "Bowtie2";
    if (has("@pg\tid:star")) return "STAR";
    if (has("bwa")) return "BWA";
    if (has("minimap2")) return "minimap2";
    if (has("bowtie2")) return "Bowtie2";
    if (has("star")) return "STAR";
    return "Unknown";
}
std::string reference_build(const std::string &t) {                // types.rs:100-147
    auto has = [&](const char *s) { return t.find(s) != std::string::npos; };
    if (has("AS:GRCh38") || has("GCA_000001405.15")) return "GRCh38";
    if (has("AS:GRCh37") || has("GCA_000001405.1")) return "GRCh37";
    if (has("AS:CHM13") || has("GCA_009914755.4") || has("chm13") || has("CHM13") || has("t2t") || has("T2T")) return "T2T-CHM13v2.0";
    if (has("SN:chr1") && has("LN:248387328") && has("M5:e469247288ceb332aee524caec92bb22")) return "T2T-CHM13v2.0";
    if (has("SN:chr1") && has("LN:248956422")) return "GRCh38";
    if (has("SN:1") && has("LN:249250621")) return "GRCh37";
    return "Unknown";
}

// One page-locked column batch of admitted records (clb_host_alloc): what clb_push_reads copies from asynchronously.
struct PinBatch {
    size_t n = 0, n_cigar = 0, n_qual = 0, cap_n = 0, cap_c = 0, cap_q = 0;
    int32_t *pos = nullptr; uint16_t *flag = nullptr; uint8_t *mapq = nullptr;
    uint32_t *cigar_off = nullptr, *cigar = nullptr; uint64_t *qual_off = nullptr; uint8_t *qual = nullptr;
    PinBatch() = default;
    PinBatch(const PinBatch &) = delete;
    PinBatch &operator=(const PinBatch &) = delete;
    ~PinBatch() {
        for (void *p : {(void *)pos, (void *)flag, (void *)mapq, (void *)cigar_off, (void *)cigar, (void *)qual_off, (void *)qual}) clb_host_free(p);
    }
    template <class T> static void grow(T *&p, size_t used, size_t ncap) {
        T *q = (T *)clb_host_alloc(ncap * sizeof(T));
        if (!q) die("cannot allocate page-locked host memory");
        if (p) { memcpy(q, p, used * sizeof(T)); clb_host_free(p); }
        p = q;
    }
    void reserve(size_t rn, size_t rc, size_t rq) {
        if (rn > cap_n) { grow(pos, n, rn); grow(flag, n, rn); grow(mapq, n, rn); grow(cigar_off, n + 1, rn + 1); grow(qual_off, n + 1, rn + 1); cap_n = rn; }
        if (rc > cap_c) { grow(cigar, n_cigar, rc); cap_c = rc; }
        if (rq > cap_q) { grow(qual, n_qual, rq); cap_q = rq; }
        cigar_off[0] = 0; qual_off[0] = 0;
    }
    void clear() { n = n_cigar = n_qual = 0; }
    bool fits(const BamRecordView &r) const { return n + 1 <= cap_n && n_cigar + r.n_cigar <= cap_c && n_qual + (size_t)std::max(0, r.l_seq) <= cap_q; }
    void push(const BamRecordView &r) {
        const size_t lq = (size_t)std::max(0, r.l_seq);
        pos[n] = r.pos; flag[n] = r.flag; mapq[n] = r.mapq;
        memcpy(cigar + n_cigar, r.cigar, 4 * (size_t)r.n_cigar); n_cigar += r.n_cigar;
        memcpy(qual + n_qual, r.qual, lq); n_qual += lq;
        n++;
        cigar_off[n] = (uint32_t)n_cigar; qual_off[n] = n_qual;
    }
};

// QNAMEs of the admitted records of one contig that reach >= 1 column, bucketed by hash: the exact distinct count
// (contig_profiler.rs:59-62) is a sort + compare per bucket, buckets in parallel.
struct NameStore {
    static constexpr unsigned kBuckets = 64;
    struct Ent { uint64_t hash; uint64_t off; uint32_t len; };
    std::vector<char> arena;
    std::vector<Ent> bucket[kBuckets];
    static uint64_t fnv(const char *p, size_t n) { uint64_t h = 1469598103934665603ull; for (size_t i = 0; i < n; i++) { h ^= (uint8_t)p[i]; h *= 1099511628211ull; } return h ^ (h >> 29); }
    void add(const char *p, uint32_t n) {
        const uint64_t h = fnv(p, n);
        bucket[h >> 58].push_back({h, arena.size(), n});
        arena.insert(arena.end(), p, p + n);
    }
    uint64_t count_unique(unsigned threads) {
        std::vector<uint64_t> cnt(kBuckets, 0);
        std::atomic<unsigned> next{0};
        auto work = [&] {
            for (;;) {
                const unsigned b = next.fetch_add(1);
                if (b >= kBuckets) break;
                auto &v = bucket[b];
                auto less = [&](const Ent &x, const Ent &y) {
                    if (x.hash != y.hash) return x.hash < y.hash;
                    const int c = memcmp(arena.data() + x.off, arena.data() + y.off, std::min(x.len, y.len));
                    return c != 0 ? c < 0 : x.len < y.len;
                };
                std::sort(v.begin(), v.end(), less);
                uint64_t n = 0;
                for (size_t i = 0; i < v.size(); i++)
                    if (i == 0 || v[i].hash != v[i - 1].hash || v[i].len != v[i - 1].len || memcmp(arena.data() + v[i].off, arena.data() + v[i - 1].off, v[i].len) != 0) n++;
                cnt[b] = n;
            }
        };
        std::vector<std::thread> th;
        for (unsigned t = 1; t < std::max(1u, std::min(threads, kBuckets)); t++) th.emplace_back(work);
        work();
        for (auto &t : th) t.join();
        uint64_t n = 0; for (uint64_t c : cnt) n += c;
        return n;
    }
};

// A queue between the two threads.  close() wakes every waiter; from then on put() drops its value and returns false, and
// take() returns false instead of blocking.
template <class T> class Channel {
  public:
    bool put(T v) {
        { std::lock_guard<std::mutex> g(m_); if (closed_) return false; q_.push_back(std::move(v)); }
        cv_.notify_one();
        return true;
    }
    bool take(T &v, double *waited_s = nullptr) {
        std::unique_lock<std::mutex> g(m_);
        const auto t0 = std::chrono::steady_clock::now();
        cv_.wait(g, [this] { return !q_.empty() || closed_; });
        if (waited_s) *waited_s += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        if (closed_) return false;
        v = std::move(q_.front()); q_.pop_front();
        return true;
    }
    void close() { { std::lock_guard<std::mutex> g(m_); closed_ = true; } cv_.notify_all(); }
  private:
    std::mutex m_; std::condition_variable cv_; std::deque<T> q_; bool closed_ = false;
};

double secs_since(std::chrono::steady_clock::time_point a) { return std::chrono::duration<double>(std::chrono::steady_clock::now() - a).count(); }

// decoder thread -> device thread: a full batch, or the end of a contig (its last batch, QNAMEs and admitted count), or an error
struct Msg { PinBatch *batch = nullptr; bool end_of_contig = false; std::unique_ptr<NameStore> names; uint64_t admitted = 0; std::string error; };

// The decoder thread: BGZF read-ahead + inflate pool (bam_reader.hpp) -> record scan -> htslib admission, one record at a time
// (clb_admitter_*) -> admitted records packed into page-locked column batches + QNAME store, handed to the device thread.
// It owns the thread, the three batches and both channels, and borrows the reader, the index (nullptr: scan the file from the
// start) and the contig list (tid, length), which must outlive it.  Closing the channels is the stop request: a blocked take()
// returns, the next hand-over fails and the thread returns.  The destructor closes them and joins, so a failure on the device
// thread (an exception unwinding past this object) cannot leave the decoder running.
class DecodeStage {
  public:
    DecodeStage(BamReader &bam, const BaiIndex *bai, const std::vector<std::pair<int32_t, uint32_t>> &contigs, uint32_t maxcnt, size_t batch_reads)
        : bam_(bam), bai_(bai), contigs_(contigs), maxcnt_(maxcnt) {
        for (auto &b : pool_) { b.reserve(batch_reads, 2 * batch_reads, 160 * batch_reads); free_.put(&b); }
        thread_ = std::thread([this] { run(); });
    }
    ~DecodeStage() { free_.close(); ready_.close(); if (thread_.joinable()) thread_.join(); }
    DecodeStage(const DecodeStage &) = delete;
    DecodeStage &operator=(const DecodeStage &) = delete;

    Msg take(double *waited_s) { Msg m; if (!ready_.take(m, waited_s)) m.error = "the decoder stopped"; return m; }
    void give_back(PinBatch *b) { free_.put(b); }
    void join() { thread_.join(); }   // after the last end-of-contig message; the timings below are final from then on
    double total_s = 0, waited_for_batch_s = 0, admission_s = 0;

  private:
    void run() {
        const auto t_start = std::chrono::steady_clock::now();
        const uint64_t tick_start = ticks();
        try {
            scan();
        } catch (const std::exception &e) {
            Msg m; m.error = e.what(); m.end_of_contig = true; ready_.put(std::move(m));
        }
        total_s = secs_since(t_start);
        admission_s = total_s > 0 ? (double)admit_ticks_ * total_s / (double)std::max<uint64_t>(1, ticks() - tick_start) : 0.0;
    }
    bool next_free(PinBatch *&b) {
        if (!free_.take(b, &waited_for_batch_s)) return false;
        b->clear();
        return true;
    }
    void scan() {
        BamRecordView rec; bool have = bai_ ? false : bam_.next(rec);
        for (const auto &[tid, clen] : contigs_) {                        // ascending tid (api/coverage.rs:229-235)
            if (bai_) {
                have = bai_->first[(size_t)tid] != UINT64_MAX;
                if (have) { bam_.seek(bai_->first[(size_t)tid]); have = bam_.next(rec); }
            }
            while (have && (rec.tid < tid && rec.tid >= 0)) have = bam_.next(rec);   // records of contigs that were not selected
            const std::unique_ptr<clb_admitter, decltype(&clb_admitter_free)> adm(clb_admitter_new(tid, maxcnt_), clb_admitter_free);
            auto names = std::make_unique<NameStore>();
            PinBatch *cur = nullptr; uint64_t admitted = 0;
            while (have && rec.tid == tid) {
                const uint64_t ta = ticks();
                const int k = clb_admitter_push(adm.get(), rec.pos, rec.flag, rec.cigar, rec.n_cigar);
                admit_ticks_ += ticks() - ta;
                if (k < 0) die("Error processing contig: records are not coordinate sorted");
                if (k == 1) {
                    if (!cur && !next_free(cur)) return;
                    if (!cur->fits(rec)) {
                        if (cur->n) { Msg m; m.batch = cur; if (!ready_.put(std::move(m)) || !next_free(cur)) return; }
                        if (!cur->fits(rec)) cur->reserve(std::max<size_t>(cur->cap_n, 1), std::max<size_t>(cur->cap_c, 2 * (size_t)rec.n_cigar),
                                                          std::max<size_t>(cur->cap_q, 2 * (size_t)std::max(0, rec.l_seq)));
                    }
                    cur->push(rec); admitted++;
                    uint64_t span = 0;
                    for (uint32_t c = 0; c < rec.n_cigar; c++) { const uint32_t op = rec.cigar[c] & 15; if ((0x18du >> op) & 1u) span += rec.cigar[c] >> 4; }
                    if (span && (uint32_t)rec.pos < clen) names->add(rec.qname, rec.l_qname ? rec.l_qname - 1 : 0);
                }
                have = bam_.next(rec);
            }
            Msg m; m.batch = cur; m.end_of_contig = true; m.names = std::move(names); m.admitted = admitted;
            if (!ready_.put(std::move(m))) return;
        }
    }

    BamReader &bam_;
    const BaiIndex *bai_;
    const std::vector<std::pair<int32_t, uint32_t>> &contigs_;
    const uint32_t maxcnt_;
    uint64_t admit_ticks_ = 0;   // per-record timing with the cycle counter (a clock call per record would cost more than the admission)
    PinBatch pool_[3];
    Channel<PinBatch *> free_;
    Channel<Msg> ready_;
    std::thread thread_;
};

struct Options {
    std::string bam, reference, out_bed = "callable_regions.bed", summary = "summary.html", templates;
    std::vector<std::string> contigs; bool have_contigs = false;
    clb_options o{4, 500, 10, 10, 20, 1, 0, 0.1};
    unsigned threads = std::max(1u, std::thread::hardware_concurrency());
    int device = 0;
    bool verbose = false, progress = false; std::string timing_json;
    std::string depth_hist; uint32_t depth_hist_max = 1000;      // --depth-histogram FILE: rows for depths 0 .. depth_hist_max (last: >=)
    std::string depth_tiles; uint32_t depth_tile_size = 1000;    // --depth-tiles FILE: one row per tile of depth_tile_size positions
    std::string depth_bedgraph;                                  // --depth-bedgraph FILE: runs of equal raw depth of every position
};

void usage() {
    fprintf(stderr, "Usage: decodingus-tools-b200 coverage <BAM_FILE> -r <REFERENCE> [-o callable_regions.bed] [-s summary.html] [-L contig]...\n"
                    "       [--min-depth 4] [--max-depth 500] [--min-mapping-quality 10] [--min-base-quality 20]\n"
                    "       [--min-depth-for-low-mapq 10] [--max-low-mapq 1] [--max-low-mapq-fraction 0.1] [--threads N] [--device D]\n"
                    "       [--report-templates DIR] [--verbose] [--progress] [--timing-json FILE]\n"
                    "       [--depth-histogram FILE] [--depth-histogram-max 1000] [--depth-tiles FILE] [--depth-tile-size 1000]\n"
                    "       [--depth-bedgraph FILE]\n");
    exit(2);
}

Options parse_options(int argc, char **argv) {
    if (argc < 3 || strcmp(argv[1], "coverage") != 0) usage();
    Options opt;
    for (int i = 2; i < argc; i++) {
        std::string a = argv[i];
        auto val = [&]() -> std::string { if (i + 1 >= argc) usage(); return argv[++i]; };
        if (a == "-r" || a == "--reference") opt.reference = val();
        else if (a == "-o" || a == "--output") opt.out_bed = val();
        else if (a == "-s" || a == "--summary") opt.summary = val();
        else if (a == "-L" || a == "--contig") { opt.contigs.push_back(val()); opt.have_contigs = true; }
        else if (a == "--min-depth") opt.o.min_depth = (uint32_t)std::stoul(val());
        else if (a == "--max-depth") opt.o.max_depth = (uint32_t)std::stoul(val());
        else if (a == "--min-mapping-quality") opt.o.min_mapping_quality = (uint8_t)std::stoul(val());
        else if (a == "--min-base-quality") opt.o.min_base_quality = (uint8_t)std::stoul(val());
        else if (a == "--min-depth-for-low-mapq") opt.o.min_depth_for_low_mapq = (uint32_t)std::stoul(val());
        else if (a == "--max-low-mapq") opt.o.max_low_mapq = (uint8_t)std::stoul(val());
        else if (a == "--max-low-mapq-fraction") opt.o.max_low_mapq_fraction = std::stod(val());
        else if (a == "--threads") opt.threads = (unsigned)std::stoul(val());
        else if (a == "--device") opt.device = std::stoi(val());
        else if (a == "--report-templates") opt.templates = val();
        else if (a == "--verbose") opt.verbose = true;
        else if (a == "--progress") opt.progress = true;
        else if (a == "--timing-json") opt.timing_json = val();
        else if (a == "--depth-histogram") opt.depth_hist = val();
        else if (a == "--depth-histogram-max") {
            const unsigned long d = std::stoul(val());
            if (d < 1 || d > 65535) usage();
            opt.depth_hist_max = (uint32_t)d;
        }
        else if (a == "--depth-tiles") opt.depth_tiles = val();
        else if (a == "--depth-bedgraph") opt.depth_bedgraph = val();
        else if (a == "--depth-tile-size") {
            const unsigned long long l = std::stoull(val());
            if (l < 256 || l > (1ull << 31)) usage();
            opt.depth_tile_size = (uint32_t)l;
        }
        else if (!a.empty() && a[0] != '-' && opt.bam.empty()) opt.bam = a;
        else usage();
    }
    if (opt.bam.empty() || opt.reference.empty()) usage();
    return opt;
}

// --progress: the reference API's ProgressEvent stream (api/mod.rs:12-18, emitted by CoverageAnalyzer::analyze at
// api/coverage.rs:40-48), one serde-style JSON object per line on stderr; Progress counts finished contigs
void progress(const Options &opt, const char *kind, const std::string &extra = "") {
    if (opt.progress) fprintf(stderr, "{\"%s\":{\"task\":\"Coverage Analysis\"%s}}\n", kind, extra.c_str());
}

// --depth-histogram: "#contig\tdepth\traw_bases\tqc_bases", then per contig one row per depth from 0 to its last non-zero bin
// (the last bin of the histogram counts that depth or more), and last the sum over all contigs under the name "*".
struct DepthHistTsv {
    std::string text = "#contig\tdepth\traw_bases\tqc_bases\n";
    std::vector<uint64_t> raw_total, qc_total;
    void add_rows(const std::string &name, const uint64_t *raw, const uint64_t *qc, uint32_t n) {
        uint32_t last = n;
        while (last > 0 && raw[last - 1] == 0 && qc[last - 1] == 0) last--;
        for (uint32_t d = 0; d < last; d++)
            text += name + "\t" + std::to_string(d) + "\t" + std::to_string(raw[d]) + "\t" + std::to_string(qc[d]) + "\n";
    }
    void add_contig(const std::string &name, const uint64_t *raw, const uint64_t *qc, uint32_t n) {
        raw_total.resize(n, 0); qc_total.resize(n, 0);
        for (uint32_t d = 0; d < n; d++) { raw_total[d] += raw[d]; qc_total[d] += qc[d]; }
        add_rows(name, raw, qc, n);
    }
    std::string finish() { add_rows("*", raw_total.data(), qc_total.data(), (uint32_t)raw_total.size()); return text; }
};

// --depth-tiles: "#contig\tstart\tend\tterritory\tcallable\tmean_raw\tmean_qc", then one row per tile, contigs in tid order.
// start / end: the tile's 0-based half-open range; mean_raw / mean_qc: depth sums over territory (0.00 when it is 0).
struct DepthTilesTsv {
    std::string text = "#contig\tstart\tend\tterritory\tcallable\tmean_raw\tmean_qc\n";
    void add_contig(const std::string &name, uint32_t contig_len, uint32_t tile_len, const uint64_t *territory, const uint64_t *callable,
                    const uint64_t *raw_sum, const uint64_t *qc_sum, uint32_t n) {
        char buf[160];
        for (uint32_t t = 0; t < n; t++) {
            const uint64_t start = (uint64_t)t * tile_len, end = std::min<uint64_t>(start + tile_len, contig_len), ter = territory[t];
            snprintf(buf, sizeof buf, "\t%llu\t%llu\t%llu\t%llu\t%.2f\t%.2f\n", (unsigned long long)start, (unsigned long long)end,
                     (unsigned long long)ter, (unsigned long long)callable[t], ter ? (double)raw_sum[t] / (double)ter : 0.0,
                     ter ? (double)qc_sum[t] / (double)ter : 0.0);
            text += name; text += buf;
        }
    }
};

bool write_file(const std::string &path, const std::string &data) {
    FILE *f = fopen(path.c_str(), "wb");
    if (!f) return false;
    const bool ok = fwrite(data.data(), 1, data.size(), f) == data.size();
    return fclose(f) == 0 && ok;
}

// What the contig loop measured, for the stderr summary line and --timing-json.
struct Timing {
    double wall_s = 0, decode_total_s = 0, decode_wait_s = 0, admit_s = 0;
    double device_ms = 0, h2d_ms = 0, bed_s = 0, names_s = 0, ref_s = 0, device_wait_s = 0;
    uint64_t total_admitted = 0, total_cells = 0;
};

// The pipeline over the selected contigs:
// decoder thread: DecodeStage
// this thread   : clb_begin_contig / clb_push_reads per batch (copies overlap the kernels of earlier windows and the
//                 decoding of the next batch) / clb_finish_contig, BED text, plots
Timing process_contigs(const Options &opt, BamReader &bam, const BaiIndex *bai, const std::map<std::string, FaiEntry> &fai,
                       std::map<int32_t, ContigStats> &stats, uint32_t largest, clb_ctx *ctx, clb_bed_writer *bed, DepthHistTsv *hist,
                       DepthTilesTsv *tiles, clb_bedgraph_writer *bedgraph) {
    auto check = [&](int rc, const char *what) { if (rc != 0) die(std::string("Error processing contig: ") + what + ": " + clb_last_error(ctx)); };
    // coverage plots land next to the BED file (callable_profiler.rs:24-27,80-83)
    const size_t slash = opt.out_bed.find_last_of('/');
    const std::string out_dir = slash == std::string::npos ? "" : opt.out_bed.substr(0, slash + 1);
    const uint32_t maxcnt = opt.o.max_depth > 0 ? opt.o.max_depth : 500;
    const auto wall0 = std::chrono::steady_clock::now();
    // batches of about a million reads for real inputs, small ones for small files (page-locking memory is not free)
    size_t kBatchReads = 1u << 20;
    {
        FILE *fsz = fopen(opt.bam.c_str(), "rb");
        if (fsz) { fseeko(fsz, 0, SEEK_END); const off_t sz = ftello(fsz); fclose(fsz); if (sz < (off_t)(256u << 20)) kBatchReads = std::max<size_t>(4096, (size_t)sz / 64); }
    }
    std::vector<std::pair<int32_t, uint32_t>> contigs;
    for (auto &kv : stats) contigs.emplace_back(kv.first, (uint32_t)kv.second.length);
    Timing t;
    {
        DecodeStage decoder(bam, bai, contigs, maxcnt, kBatchReads);
        size_t contigs_done = 0;
        for (auto &kv : stats) {
            ContigStats &st = kv.second;
            const uint32_t clen = (uint32_t)st.length;
            const auto tr = std::chrono::steady_clock::now();
            std::vector<uint8_t> ref;
            auto fe = fai.find(st.name);
            if (fe != fai.end()) ref = load_contig(opt.reference, fe->second);   // missing contig / short sequence reads as 'N'
            t.ref_s += secs_since(tr);
            check(clb_begin_contig(ctx, kv.first, st.name.c_str(), clen, ref.data(), ref.size(), 0, largest, 0, clen, 0), "begin");
            std::unique_ptr<NameStore> names; uint64_t admitted = 0;
            for (;;) {
                Msg m = decoder.take(&t.device_wait_s);
                if (!m.error.empty()) die(m.error);
                if (m.batch) {
                    if (m.batch->n) {
                        clb_read_batch rb{m.batch->n, m.batch->n_cigar, m.batch->n_qual, m.batch->pos, m.batch->flag, m.batch->mapq,
                                          m.batch->cigar_off, m.batch->cigar, m.batch->qual_off, m.batch->qual};
                        check(clb_push_reads(ctx, &rb), "push");
                        check(clb_wait_uploads(ctx), "upload");                  // the batch's buffers go back to the decoder
                    }
                    decoder.give_back(m.batch);
                }
                if (m.end_of_contig) { names = std::move(m.names); admitted = m.admitted; break; }
            }
            clb_contig_result res{};
            check(clb_finish_contig(ctx, &res), "finish");
            t.device_ms += res.kernel_ms; t.h2d_ms += res.h2d_ms;
            const auto tn = std::chrono::steady_clock::now();
            st.n_reads = names->count_unique(opt.threads);
            names.reset();
            t.names_s += secs_since(tn);
            for (int s = 0; s < 6; s++) st.counts[s] = res.state_counts[s];
            st.n_covered = res.n_covered_bases; st.sum_cov = res.summed_coverage; st.sum_bq = res.summed_baseq;
            st.sum_mapq = res.summed_mapq; st.qbases = res.quality_bases;
            t.total_admitted += admitted; t.total_cells += res.summed_coverage;
            if (hist) {
                const uint64_t *raw = nullptr, *qc = nullptr; uint32_t n = 0;
                check(clb_depth_histogram(ctx, &raw, &qc, &n), "depth histogram");
                hist->add_contig(st.name, raw, qc, n);
            }
            if (tiles) {
                const uint64_t *ter = nullptr, *cal = nullptr, *raw = nullptr, *qc = nullptr; uint32_t n = 0, len = 0;
                check(clb_depth_tiles(ctx, &ter, &cal, &raw, &qc, &n, &len), "depth tiles");
                tiles->add_contig(st.name, clen, len, ter, cal, raw, qc, n);
            }
            const auto tb = std::chrono::steady_clock::now();
            std::vector<uint32_t> bins(res.bins, res.bins + 3 * (size_t)res.n_bins);
            int has_bins = 0;
            const int rc = clb_bed_writer_add_contig(bed, st.name.c_str(), clen, res.intervals, res.n_intervals, bins.data(), res.n_bins, res.stride, &has_bins);
            if (rc == CLB_E_IO) die("Error processing contig: cannot write " + opt.out_bed);
            if (rc != 0) die("Error processing contig: interval list does not tile the contig");
            if (bedgraph) {
                const clb_depth_run *runs = nullptr; uint64_t n = 0;
                check(clb_depth_runs(ctx, &runs, &n), "depth runs");
                const int rg = clb_bedgraph_writer_add_contig(bedgraph, st.name.c_str(), clen, runs, n);
                if (rg == CLB_E_IO) die("cannot write " + opt.depth_bedgraph);
                if (rg != 0) die("Error processing contig: depth runs do not tile the contig");
            }
            if (has_bins && res.stride) {                                        // finish_contig, callable_profiler.rs:64-86
                const std::string path = out_dir + st.name + "_coverage.svg";
                if (!write_file(path, report::render_coverage_svg(st.name, clen, res.stride, bins.data(), res.n_bins)))
                    die("Error processing contig: cannot create " + path);
            }
            t.bed_s += secs_since(tb);
            if (opt.verbose)
                fprintf(stderr, "%s: %llu admitted reads, %llu cells, %.2f ms on device\n", st.name.c_str(), (unsigned long long)admitted,
                        (unsigned long long)res.summed_coverage, res.kernel_ms);
            progress(opt, "Progress", ",\"current\":" + std::to_string(++contigs_done) + ",\"total\":" + std::to_string(stats.size()));
        }
        decoder.join();
        t.decode_total_s = decoder.total_s; t.decode_wait_s = decoder.waited_for_batch_s; t.admit_s = decoder.admission_s;
    }   // the batches are freed here, inside the wall time
    t.wall_s = secs_since(wall0);
    return t;
}

void report_timing(const Options &opt, const Timing &t, size_t n_contigs, double inflate_s) {
    fprintf(stderr, "coverage: %zu contigs, %llu admitted reads, %llu aligned bases | wall %.3f s | host decode %.3f s (BGZF inflate %.3f s on %u threads, "
                    "admission %.3f s inline, waiting for a free batch %.3f s) | device %.3f s kernels, %.3f s H2D | reference load %.3f s | "
                    "unique names %.3f s | BED + plots %.3f s | device thread waited %.3f s for the decoder\n",
            n_contigs, (unsigned long long)t.total_admitted, (unsigned long long)t.total_cells, t.wall_s, t.decode_total_s - t.decode_wait_s,
            inflate_s, opt.threads, t.admit_s, t.decode_wait_s, t.device_ms * 1e-3, t.h2d_ms * 1e-3, t.ref_s, t.names_s, t.bed_s, t.device_wait_s);
    if (!opt.timing_json.empty()) {
        FILE *ft = fopen(opt.timing_json.c_str(), "wb");
        if (ft) {
            fprintf(ft, "{\"contigs\": %zu, \"admitted_reads\": %llu, \"aligned_bases\": %llu, \"wall_s\": %.6f, \"decode_s\": %.6f, \"inflate_s\": %.6f, "
                        "\"threads\": %u, \"admission_s\": %.6f, \"decoder_waited_for_batch_s\": %.6f, \"device_kernels_s\": %.6f, \"h2d_s\": %.6f, "
                        "\"reference_load_s\": %.6f, \"unique_names_s\": %.6f, \"bed_and_plots_s\": %.6f, \"device_thread_waited_s\": %.6f}\n",
                    n_contigs, (unsigned long long)t.total_admitted, (unsigned long long)t.total_cells, t.wall_s, t.decode_total_s - t.decode_wait_s, inflate_s,
                    opt.threads, t.admit_s, t.decode_wait_s, t.device_ms * 1e-3, t.h2d_ms * 1e-3, t.ref_s, t.names_s, t.bed_s, t.device_wait_s);
            fclose(ft);
        }
    }
}

// build_coverage_export (report.rs:15-134): writes summary.json and returns what the HTML page shows (the summary; rows gets
// one row per contig in natural order)
report::Summary write_summary_json(const Options &opt, const std::string &header_text, const report::BamStats &bs,
                                   const std::map<int32_t, ContigStats> &stats, std::vector<report::ContigRow> &rows) {
    std::vector<const ContigStats *> order;
    for (auto &kv : stats) order.push_back(&kv.second);
    std::stable_sort(order.begin(), order.end(), [](const ContigStats *a, const ContigStats *b) { return contig_less(a->name, b->name); });
    uint64_t total_bases = 0, callable = 0, q30_bases = 0, total_qpos = 0, total_unique = 0;
    double total_depth = 0, total_mapq = 0, total_baseq = 0;
    std::string cj;
    auto exists = [](const std::string &p) { FILE *f = fopen(p.c_str(), "rb"); if (f) fclose(f); return f != nullptr; };
    for (size_t i = 0; i < order.size(); i++) {
        const ContigStats &s = *order[i];
        const double amq = s.qbases ? (double)s.sum_mapq / (double)s.qbases : 0.0, abq = s.qbases ? (double)s.sum_bq / (double)s.qbases : 0.0;
        const double q30 = s.qbases ? (abq >= 30.0 ? 100.0 : abq < 20.0 ? 0.0 : ((abq - 20.0) / 10.0) * 100.0) : 0.0;
        const double covp = s.length ? ((double)s.n_covered / (double)s.length) * 100.0 : 0.0;
        const double adep = s.n_covered ? (double)s.sum_cov / (double)s.n_covered : 0.0;
        total_bases += s.length; callable += s.counts[CLB_CALLABLE];
        total_depth += adep * (double)s.length; total_mapq += amq * (double)s.length; total_baseq += abq * (double)s.length;
        q30_bases += (uint64_t)(q30 / 100.0 * (double)s.length); total_qpos += s.length; total_unique += (uint32_t)s.n_reads;
        report::ContigRow row{s.name, s.length, s.n_reads, s.n_covered, covp, adep, amq, abq, q30, {0, 0, 0, 0, 0, 0},
                              exists(s.name + "_coverage.svg")};   // path relative to the CWD, as report.rs:318-319 tests it
        for (int k = 0; k < 6; k++) row.counts[k] = s.counts[k];
        rows.push_back(row);
        cj += std::string(i ? ",\n" : "") + "      {\n        \"name\": " + jstr(s.name) + ",\n        \"length\": " + std::to_string(s.length) +
              ",\n        \"unique_reads\": " + std::to_string(s.n_reads) + ",\n        \"coverage_percent\": " + fmt_f64(covp) +
              ",\n        \"average_depth\": " + fmt_f64(adep) + ",\n        \"covered_bases\": " + std::to_string(s.n_covered) +
              ",\n        \"total_bases\": " + std::to_string(s.length) + ",\n        \"quality_stats\": {\n          \"average_mapq\": " + fmt_f64(amq) +
              ",\n          \"average_baseq\": " + fmt_f64(abq) + ",\n          \"q30_percentage\": " + fmt_f64(q30) +
              "\n        },\n        \"state_distribution\": {\n          \"ref_n\": " + std::to_string(s.counts[0]) + ",\n          \"callable\": " +
              std::to_string(s.counts[1]) + ",\n          \"no_coverage\": " + std::to_string(s.counts[2]) + ",\n          \"low_coverage\": " +
              std::to_string(s.counts[3]) + ",\n          \"excessive_coverage\": " + std::to_string(s.counts[4]) +
              ",\n          \"poor_mapping_quality\": " + std::to_string(s.counts[5]) + "\n        }\n      }";
    }
    const double avg_depth = total_bases ? total_depth / (double)total_bases : 0.0;
    const double call_pct = total_bases ? ((double)callable / (double)total_bases) * 100.0 : 0.0;
    // collect_coverage_plots (api/coverage.rs:262-275): plots found in the CWD; the reference lists them in HashMap order, here by tid
    std::string plots;
    for (auto &kv : stats) {
        const std::string p = kv.second.name + "_coverage.svg";
        if (exists(p)) plots += std::string(plots.empty() ? "\n      " : ",\n      ") + jstr(p);
    }
    if (!plots.empty()) plots += "\n    ";
    std::string js = "{\n  \"export\": {\n    \"summary\": {\n      \"aligner\": " + jstr(detect_aligner(header_text)) + ",\n      \"reference_build\": " +
        jstr(reference_build(header_text)) + ",\n      \"sequencing_platform\": " + jstr(bs.infer_platform()) + ",\n      \"read_length\": " + std::to_string(bs.average_read_length()) +
        ",\n      \"total_bases\": " + std::to_string(total_bases) + ",\n      \"callable_bases\": " + std::to_string(callable) +
        ",\n      \"callable_percentage\": " + fmt_f64(call_pct) + ",\n      \"average_depth\": " + fmt_f64(avg_depth) + ",\n      \"contigs_analyzed\": " +
        std::to_string(stats.size()) + "\n    },\n    \"contigs\": [" + (order.empty() ? "" : "\n" + cj + "\n    ") + "],\n    \"quality_metrics\": {\n      \"average_mapq\": " +
        fmt_f64(total_qpos ? total_mapq / (double)total_qpos : 0.0) + ",\n      \"average_baseq\": " + fmt_f64(total_qpos ? total_baseq / (double)total_qpos : 0.0) +
        ",\n      \"q30_percentage\": " + fmt_f64(total_qpos ? ((double)q30_bases / (double)total_qpos) * 100.0 : 0.0) + "\n    },\n    \"total_unique_reads\": " +
        std::to_string(total_unique) + "\n  },\n  \"files\": {\n    \"bed_file\": " + jstr(opt.out_bed) + ",\n    \"summary_html\": " + jstr(opt.summary) +
        ",\n    \"coverage_plots\": [" + plots + "]\n  }\n}";
    if (!write_file("summary.json", js)) die("cannot create summary.json");   // main.rs:68: always in the CWD
    return report::Summary{reference_build(header_text), detect_aligner(header_text), bs.infer_platform(), bs.average_read_length(), total_unique, total_bases,
                           callable, (uint64_t)stats.size(), bs.max_samples, call_pct, avg_depth, total_qpos ? total_mapq / (double)total_qpos : 0.0,
                           total_qpos ? total_baseq / (double)total_qpos : 0.0};
}

// write_html_report (report.rs:136-160)
void write_html_report(const Options &opt, const report::Summary &sm, const std::vector<report::ContigRow> &rows) {
    auto slurp = [](const std::string &p) { std::ifstream f(p, std::ios::binary); if (!f) die("cannot read " + p); return std::string((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>()); };
    const std::string header = opt.templates.empty() ? report::default_header() : slurp(opt.templates + "/report_header.html");
    const std::string footer = opt.templates.empty() ? report::default_footer() : slurp(opt.templates + "/report_footer.html");
    if (!write_file(opt.summary, report::render_html_report(sm, rows, header, footer))) die("cannot create " + opt.summary);
}

int run(int argc, char **argv) {
    const Options opt = parse_options(argc, argv);
    BamReader bam(opt.bam, opt.threads);
    const BamHeader &H = bam.header();
    const auto fai = load_fai(opt.reference);

    // initialize_contig_stats + validate_contig_selection (api/coverage.rs:149-204)
    std::set<std::string> selected(opt.contigs.begin(), opt.contigs.end());
    std::map<int32_t, ContigStats> stats;
    for (size_t tid = 0; tid < H.names.size(); tid++) {
        if (opt.have_contigs && !selected.count(H.names[tid])) continue;
        ContigStats s; s.name = H.names[tid]; s.length = H.lens[tid];
        stats[(int32_t)tid] = s;
    }
    if (opt.have_contigs && stats.empty()) {
        std::string l; for (size_t i = 0; i < opt.contigs.size(); i++) l += (i ? ", " : "") + opt.contigs[i];
        die("None of the specified contigs (" + l + ") were found in the BAM file");
    }
    uint32_t largest = 0;                                               // initialize_counter (api/coverage.rs:206-219)
    for (auto &kv : stats) if (kv.second.name != "chrM") largest = std::max<uint32_t>(largest, (uint32_t)kv.second.length);

    char err[512];
    std::unique_ptr<clb_ctx, decltype(&clb_destroy)> ctx(clb_create(opt.device, &opt.o, err, sizeof err), clb_destroy);
    if (!ctx) die(std::string("GPU context: ") + err);
    if (!opt.depth_hist.empty() && clb_set_depth_histogram(ctx.get(), opt.depth_hist_max + 1) != 0)
        die(std::string("GPU context: ") + clb_last_error(ctx.get()));
    if (!opt.depth_tiles.empty() && clb_set_depth_tiles(ctx.get(), opt.depth_tile_size) != 0)
        die(std::string("GPU context: ") + clb_last_error(ctx.get()));
    if (!opt.depth_bedgraph.empty() && clb_set_depth_runs(ctx.get(), 1) != 0)
        die(std::string("GPU context: ") + clb_last_error(ctx.get()));
    std::unique_ptr<clb_bed_writer, decltype(&clb_bed_writer_close)> bed(clb_bed_writer_open(opt.out_bed.c_str(), largest), clb_bed_writer_close);
    if (!bed) die("Failed to create CallableProfiler: cannot create " + opt.out_bed);
    // opened before the first contig (a FIFO blocks here until its reader is there), written per contig after its BED lines
    std::unique_ptr<clb_bedgraph_writer, decltype(&clb_bedgraph_writer_close)> bedgraph(nullptr, clb_bedgraph_writer_close);
    if (!opt.depth_bedgraph.empty()) {
        bedgraph.reset(clb_bedgraph_writer_open(opt.depth_bedgraph.c_str()));
        if (!bedgraph) die("cannot write " + opt.depth_bedgraph);
    }

    // BamStats: its own pass over the first 10 000 records of the file, primary alignments only (bam_stats.rs:44-76)
    report::BamStats bs;
    {
        BamReader head(opt.bam, std::min(opt.threads, 4u));
        BamRecordView r;
        while (!bs.full() && head.next(r)) bs.add_record(std::string(r.qname, r.l_qname ? r.l_qname - 1 : 0), r.flag, (uint64_t)std::max(0, r.l_seq));
    }
    // With a contig selection and a .bai next to the BAM the reader jumps to each contig (what bam.fetch does, mod.rs:54);
    // otherwise the coordinate-sorted file is scanned once from the start.
    BaiIndex bai;
    const bool indexed = opt.have_contigs && load_bai(opt.bam, bai) && bai.first.size() == H.names.size();

    progress(opt, "Started");
    try {
        DepthHistTsv hist;
        DepthTilesTsv tiles;
        const Timing t = process_contigs(opt, bam, indexed ? &bai : nullptr, fai, stats, largest, ctx.get(), bed.get(),
                                         opt.depth_hist.empty() ? nullptr : &hist, opt.depth_tiles.empty() ? nullptr : &tiles, bedgraph.get());
        report_timing(opt, t, stats.size(), bam.inflate_seconds());
        if (clb_bed_writer_close(bed.release()) != 0) die("failed to write " + opt.out_bed);
        if (bedgraph && clb_bedgraph_writer_close(bedgraph.release()) != 0) die("cannot write " + opt.depth_bedgraph);
        if (!opt.depth_hist.empty() && !write_file(opt.depth_hist, hist.finish())) die("cannot write " + opt.depth_hist);
        if (!opt.depth_tiles.empty() && !write_file(opt.depth_tiles, tiles.text)) die("cannot write " + opt.depth_tiles);
        ctx.reset();
        std::vector<report::ContigRow> rows;
        const report::Summary sm = write_summary_json(opt, H.text, bs, stats, rows);
        write_html_report(opt, sm, rows);
    } catch (const std::exception &e) {
        progress(opt, "Error", ",\"error\":" + jstr(e.what()));
        throw;
    }
    progress(opt, "Completed");
    return 0;
}

}  // namespace

int main(int argc, char **argv) {
    try {
        return run(argc, argv);
    } catch (const std::exception &e) {      // every failure: message + exit code 1, the partially written BED stays behind
        fprintf(stderr, "Error: %s\n", e.what());
        return 1;
    }
}
