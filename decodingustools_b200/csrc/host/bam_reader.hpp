// bam_reader.hpp -- what rust-htslib does for the reference's `coverage` command, for this host: multi-threaded BGZF inflate,
// a sequential BAM record scan (the file is coordinate sorted, no .bai needed) and .fai-indexed FASTA contig loads.
//
// Reference call sites this stands in for: BamReaderFactory::open / open_indexed (src/utils/bam_reader.rs:7-35),
// bam.fetch + records (src/callable_loci/mod.rs:54-55, profilers/bam_stats.rs:52-66), faidx::Reader::fetch_seq
// (mod.rs:79,100,128).  Like htslib, records whose CIGAR has more than 65535 ops are stored with a placeholder CIGAR
// (<l_seq>S<ref_len>N) and the real one in a CG:B,I tag; next() hands out the real one.
// Errors are thrown as std::runtime_error (the CLI prints them as "Error: ..." and exits 1, as the reference does).
#pragma once
#include <zlib.h>

#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <deque>
#include <fstream>
#include <functional>
#include <map>
#include <mutex>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

namespace bamio {

[[noreturn]] inline void die(const std::string &m) { throw std::runtime_error(m); }

// ------------------------------------------------------------------------------------------------ BGZF / BAM
struct BamHeader { std::string text; std::vector<std::string> names; std::vector<uint32_t> lens; };

struct BamRecordView {
    int32_t tid, pos; uint8_t mapq; uint16_t flag; uint32_t n_cigar; int32_t l_seq;
    const char *qname; uint32_t l_qname; const uint32_t *cigar; const uint8_t *qual;
};

// N worker threads that live as long as the stream: run(fn) executes fn(t) on every worker and returns when all are done.
class WorkerPool {
  public:
    explicit WorkerPool(unsigned n) : n_(std::max(1u, n)) {
        for (unsigned t = 0; t < n_; t++) th_.emplace_back([this, t] { loop(t); });
    }
    ~WorkerPool() {
        { std::lock_guard<std::mutex> g(m_); stop_ = true; gen_++; }
        cv_.notify_all();
        for (auto &t : th_) t.join();
    }
    unsigned size() const { return n_; }
    void run(const std::function<void(unsigned)> &fn) {
        std::unique_lock<std::mutex> g(m_);
        fn_ = &fn; pending_ = n_; gen_++;
        cv_.notify_all();
        done_.wait(g, [this] { return pending_ == 0; });
        fn_ = nullptr;
    }

  private:
    void loop(unsigned t) {
        uint64_t seen = 0;
        for (;;) {
            const std::function<void(unsigned)> *fn;
            {
                std::unique_lock<std::mutex> g(m_);
                cv_.wait(g, [&] { return gen_ != seen; });
                seen = gen_;
                if (stop_) return;
                fn = fn_;
            }
            (*fn)(t);
            { std::lock_guard<std::mutex> g(m_); if (--pending_ == 0) done_.notify_one(); }
        }
    }
    unsigned n_; std::vector<std::thread> th_; std::mutex m_; std::condition_variable cv_, done_;
    const std::function<void(unsigned)> *fn_ = nullptr; unsigned pending_ = 0; uint64_t gen_ = 0; bool stop_ = false;
};

// BGZF file -> inflated bytes.  A read-ahead thread reads compressed chunks, inflates their blocks on a persistent worker
// pool and queues the results (at most kDepth chunks ahead), so the record scan never waits for zlib when the pool keeps up.
class BgzfStream {
  public:
    BgzfStream(const std::string &path, unsigned threads) : pool_(std::max(1u, threads)) {
        fp_ = fopen(path.c_str(), "rb");
        if (!fp_) die("Failed to open BAM file: " + path);
    }
    ~BgzfStream() { stop_reader(); if (fp_) fclose(fp_); }
    // Continue at a compressed file offset (the upper 48 bits of a BAI virtual offset).  Reads start small and grow again,
    // so that fetching a small contig does not inflate 64 MB of its neighbours.
    void seek(uint64_t coffset) {
        stop_reader();
        if (fseeko(fp_, (off_t)coffset, SEEK_SET) != 0) die("seek failed in BAM file");
        chunk_ = 1u << 20;
    }
    // Hands out the next batch of inflated bytes: buf[kHeadroom ..) is the data, the kHeadroom bytes in front of it are
    // free for the caller (the record scan copies the unfinished tail of the previous batch there instead of moving the
    // batch).  Returns false at EOF.  A read or inflate failure is thrown once the batches before it have been handed out,
    // so it surfaces where the data ends, not whenever the read-ahead thread got there.
    static constexpr size_t kHeadroom = 4u << 20;
    bool next(std::vector<uint8_t> &buf) {
        if (!reader_.joinable() && !finished_) start_reader();
        std::unique_lock<std::mutex> g(m_);
        cv_.wait(g, [this] { return !q_.empty() || finished_; });
        if (q_.empty()) {
            if (!error_.empty()) { const std::string e = error_; g.unlock(); die(e); }
            return false;
        }
        buf = std::move(q_.front());
        q_.pop_front();
        g.unlock();
        cv_space_.notify_one();
        return true;
    }
    double inflate_seconds() const { return inflate_s_; }

  private:
    static constexpr size_t kChunk = 64u << 20;
    static constexpr size_t kDepth = 2;
    void start_reader() { stop_ = false; finished_ = false; reader_ = std::thread([this] { reader_loop(); }); }
    void stop_reader() {
        { std::lock_guard<std::mutex> g(m_); stop_ = true; }
        cv_space_.notify_all();
        if (reader_.joinable()) reader_.join();
        q_.clear(); finished_ = false; stop_ = false; error_.clear();
    }
    void finish(const std::string &err) {
        { std::lock_guard<std::mutex> g(m_); finished_ = true; if (!err.empty()) error_ = err; }
        cv_.notify_all();
    }
    void reader_loop() {
        std::vector<uint8_t> cbuf;
        bool eof = false;
        try {
            for (;;) {
                {
                    std::unique_lock<std::mutex> g(m_);
                    cv_space_.wait(g, [this] { return q_.size() < kDepth || stop_; });
                    if (stop_) return;
                }
                if (eof && cbuf.empty()) break;
                const size_t have = cbuf.size(), want = chunk_;
                chunk_ = std::min(kChunk, chunk_ * 4);
                cbuf.resize(have + want);
                const size_t got = eof ? 0 : fread(cbuf.data() + have, 1, want, fp_);
                cbuf.resize(have + got);
                if (got < want) eof = true;
                struct Blk { size_t off, clen, ulen, uoff; };
                std::vector<Blk> blks; size_t o = 0, utotal = 0;
                while (o + 18 <= cbuf.size()) {
                    const uint8_t *p = cbuf.data() + o;
                    if (p[0] != 0x1f || p[1] != 0x8b || p[2] != 8 || !(p[3] & 4)) die("not a BGZF file (bad block header)");
                    const uint32_t xlen = p[10] | (p[11] << 8);
                    if (o + 12 + xlen > cbuf.size()) break;
                    uint32_t bsize = 0; bool found = false;
                    for (uint32_t x = 0; x + 4 <= xlen;) {
                        const uint8_t *s = p + 12 + x; const uint32_t sl = s[2] | (s[3] << 8);
                        if (s[0] == 'B' && s[1] == 'C' && sl == 2) { bsize = (s[4] | (s[5] << 8)) + 1u; found = true; }
                        x += 4 + sl;
                    }
                    if (!found) die("BGZF block without BC field");
                    if (o + bsize > cbuf.size()) break;
                    const uint8_t *tail = p + bsize - 4;
                    const uint32_t isize = tail[0] | (tail[1] << 8) | (tail[2] << 16) | ((uint32_t)tail[3] << 24);
                    blks.push_back({o + 12 + xlen, bsize - 12 - xlen - 8, isize, utotal});
                    utotal += isize; o += bsize;
                }
                if (blks.empty() && !cbuf.empty() && eof) die("truncated BGZF file");
                std::vector<uint8_t> out(utotal ? kHeadroom + utotal : 0);
                std::vector<int> err(pool_.size(), 0);
                const auto t0 = std::chrono::steady_clock::now();
                const unsigned nt = pool_.size();
                pool_.run([&](unsigned t) {
                    z_stream zs; memset(&zs, 0, sizeof zs);
                    if (inflateInit2(&zs, -15) != Z_OK) { err[t] = 1; return; }
                    for (size_t i = t; i < blks.size(); i += nt) {
                        if (!blks[i].ulen) continue;
                        inflateReset(&zs);
                        zs.next_in = cbuf.data() + blks[i].off; zs.avail_in = (uInt)blks[i].clen;
                        zs.next_out = out.data() + kHeadroom + blks[i].uoff; zs.avail_out = (uInt)blks[i].ulen;
                        const int rc = inflate(&zs, Z_FINISH);
                        if (rc != Z_STREAM_END || zs.avail_out != 0) { err[t] = 1; break; }
                    }
                    inflateEnd(&zs);
                });
                inflate_s_ += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
                for (int e : err) if (e) die("BGZF inflate failed");
                cbuf.erase(cbuf.begin(), cbuf.begin() + (long)o);
                if (!out.empty() || (eof && cbuf.empty())) {
                    std::lock_guard<std::mutex> g(m_);
                    if (!out.empty()) q_.push_back(std::move(out));
                }
                cv_.notify_all();
                if (eof && cbuf.empty()) break;
            }
            finish("");
        } catch (const std::exception &e) {
            finish(e.what());
        }
    }
    WorkerPool pool_;
    FILE *fp_ = nullptr;
    size_t chunk_ = kChunk;
    std::thread reader_;
    std::mutex m_; std::condition_variable cv_, cv_space_;
    std::deque<std::vector<uint8_t>> q_;
    bool stop_ = false, finished_ = false; std::string error_;
    double inflate_s_ = 0;
};

class BamReader {
  public:
    BamReader(const std::string &path, unsigned threads) : bz_(path, threads) {
        need(12);
        if (memcmp(cur(), "BAM\1", 4) != 0) die("Failed to open BAM file: not a BAM (CRAM is not supported by this host)");
        const int32_t l_text = rd32(4); need(12 + (size_t)l_text);
        hdr_.text.assign((const char *)cur() + 8, (size_t)l_text);
        const int32_t n_ref = rd32(8 + l_text); off_ += 12 + (size_t)l_text;
        for (int32_t i = 0; i < n_ref; i++) {
            need(4); const int32_t l_name = rd32(0); need(8 + (size_t)l_name);
            hdr_.names.emplace_back((const char *)cur() + 4, (size_t)std::max(0, l_name - 1));
            hdr_.lens.push_back((uint32_t)rd32(4 + l_name));
            off_ += 8 + (size_t)l_name;
        }
    }
    const BamHeader &header() const { return hdr_; }
    // Continue at a BAI virtual offset (compressed block offset << 16 | offset inside the inflated block).
    void seek(uint64_t voffset) {
        bz_.seek(voffset >> 16);
        buf_.clear(); off_ = 0;
        const size_t skip = (size_t)(voffset & 0xffffu);
        if (skip && !need(skip)) die("BAI offset past the end of the BAM file");
        off_ += skip;                                                  // need() may have moved off_ to the new batch's data start
    }
    bool next(BamRecordView &r) {
        if (!need(4)) return false;
        const int32_t bs = rd32(0);
        if (bs < 32 || !need(4 + (size_t)bs)) die("truncated BAM record");
        const uint8_t *p = cur() + 4;
        auto i32 = [&](int o) { int32_t v; memcpy(&v, p + o, 4); return v; };
        auto u16 = [&](int o) { uint16_t v; memcpy(&v, p + o, 2); return v; };
        r.tid = i32(0); r.pos = i32(4); r.l_qname = p[8]; r.mapq = p[9]; r.n_cigar = u16(12); r.flag = u16(14); r.l_seq = i32(16);
        r.qname = (const char *)p + 32;
        r.cigar = (const uint32_t *)(p + 32 + r.l_qname);
        r.qual = p + 32 + r.l_qname + 4 * (size_t)r.n_cigar + ((size_t)r.l_seq + 1) / 2;
        const uint8_t *aux = r.qual + (size_t)std::max(0, r.l_seq), *end = p + bs;
        if (aux > end) die("truncated BAM record");
        // long CIGAR convention (SAM spec 4.2.2): <l_seq>S<ref_len>N placeholder + CG:B,I tag
        if (r.n_cigar == 2 && (r.cigar[0] & 15u) == 4u && (int32_t)(r.cigar[0] >> 4) == r.l_seq && (r.cigar[1] & 15u) == 3u) find_cg(aux, end, r);
        off_ += 4 + (size_t)bs;
        return true;
    }

  private:
    static size_t aux_size(uint8_t t) { return t == 'A' || t == 'c' || t == 'C' ? 1 : t == 's' || t == 'S' ? 2 : t == 'i' || t == 'I' || t == 'f' ? 4 : 0; }
    static void find_cg(const uint8_t *a, const uint8_t *end, BamRecordView &r) {
        while (a + 3 <= end) {
            const uint8_t t = a[2]; const uint8_t *v = a + 3;
            size_t len;
            if (t == 'Z' || t == 'H') { const void *z = memchr(v, 0, (size_t)(end - v)); if (!z) return; len = (size_t)((const uint8_t *)z - v) + 1; }
            else if (t == 'B') {
                if (v + 5 > end) return;
                uint32_t n; memcpy(&n, v + 1, 4);
                const size_t es = aux_size(v[0]); if (!es) return;
                if (a[0] == 'C' && a[1] == 'G' && v[0] == 'I' && v + 5 + 4 * (size_t)n <= end) { r.cigar = (const uint32_t *)(v + 5); r.n_cigar = n; return; }
                len = 5 + es * (size_t)n;
            } else { len = aux_size(t); if (!len) return; }
            a = v + len;
        }
    }
    const uint8_t *cur() const { return buf_.data() + off_; }
    int32_t rd32(size_t o) const { int32_t v; memcpy(&v, cur() + o, 4); return v; }
    bool need(size_t n) {
        while (buf_.size() - off_ < n) {
            std::vector<uint8_t> nb;
            if (!bz_.next(nb)) return false;
            const size_t tail = buf_.size() - off_;                    // unfinished bytes of the previous batch
            if (tail <= BgzfStream::kHeadroom) {                       // the usual case: park them in the new batch's headroom
                if (tail) memcpy(nb.data() + BgzfStream::kHeadroom - tail, buf_.data() + off_, tail);
                buf_.swap(nb); off_ = BgzfStream::kHeadroom - tail;
            } else {                                                   // a record larger than the headroom: join the two
                std::vector<uint8_t> j(tail + nb.size() - BgzfStream::kHeadroom);
                memcpy(j.data(), buf_.data() + off_, tail);
                memcpy(j.data() + tail, nb.data() + BgzfStream::kHeadroom, nb.size() - BgzfStream::kHeadroom);
                buf_.swap(j); off_ = 0;
            }
        }
        return true;
    }
  public:
    double inflate_seconds() const { return bz_.inflate_seconds(); }
  private:
    BgzfStream bz_; std::vector<uint8_t> buf_; size_t off_ = 0; BamHeader hdr_;
};

// ------------------------------------------------------------------------------------------------ BAI
// What `bam.fetch((tid, 0, len))` needs from the index (mod.rs:54): where the first record of a contig starts.
// first[tid] = smallest chunk start over the contig's bins (UINT64_MAX: no records).  Looks for <bam>.bai, then <stem>.bai.
struct BaiIndex { std::vector<uint64_t> first; };
inline bool load_bai(const std::string &bam_path, BaiIndex &out) {
    std::ifstream in(bam_path + ".bai", std::ios::binary);
    if (!in && bam_path.size() > 4 && bam_path.compare(bam_path.size() - 4, 4, ".bam") == 0) in.open(bam_path.substr(0, bam_path.size() - 4) + ".bai", std::ios::binary);
    if (!in) return false;
    std::vector<uint8_t> b((std::istreambuf_iterator<char>(in)), std::istreambuf_iterator<char>());
    size_t o = 0;
    auto u32 = [&]() { if (o + 4 > b.size()) die("truncated BAI index"); uint32_t v; memcpy(&v, b.data() + o, 4); o += 4; return v; };
    auto u64 = [&]() { if (o + 8 > b.size()) die("truncated BAI index"); uint64_t v; memcpy(&v, b.data() + o, 8); o += 8; return v; };
    if (b.size() < 8 || memcmp(b.data(), "BAI\1", 4) != 0) die("not a BAI index");
    o = 4;
    const uint32_t n_ref = u32();
    out.first.assign(n_ref, UINT64_MAX);
    for (uint32_t r = 0; r < n_ref; r++) {
        const uint32_t n_bin = u32();
        for (uint32_t i = 0; i < n_bin; i++) {
            const uint32_t bin = u32(), n_chunk = u32();
            for (uint32_t c = 0; c < n_chunk; c++) {
                const uint64_t beg = u64(); u64();
                if (bin != 37450u) out.first[r] = std::min(out.first[r], beg);     // 37450: the metadata pseudo-bin
            }
        }
        const uint32_t n_intv = u32();
        for (uint32_t i = 0; i < n_intv; i++) u64();
    }
    return true;
}

// ------------------------------------------------------------------------------------------------ FASTA
struct FaiEntry { uint64_t len, offset; uint32_t linebases, linewidth; };
inline std::map<std::string, FaiEntry> load_fai(const std::string &fasta) {
    std::map<std::string, FaiEntry> m;
    std::ifstream in(fasta + ".fai");
    if (!in) die("Failed to open reference: " + fasta + ".fai is missing (the reference also requires it, api/coverage.rs:73)");
    std::string name; FaiEntry e;
    while (in >> name >> e.len >> e.offset >> e.linebases >> e.linewidth) { m[name] = e; in.ignore(1 << 20, '\n'); }
    return m;
}
inline std::vector<uint8_t> load_contig(const std::string &fasta, const FaiEntry &e) {
    std::vector<uint8_t> seq; seq.reserve(e.len);
    FILE *fp = fopen(fasta.c_str(), "rb");
    if (!fp) die("Failed to open reference: " + fasta);
    const uint64_t lines = e.linebases ? (e.len + e.linebases - 1) / e.linebases : 0;
    std::vector<uint8_t> raw((size_t)(lines * e.linewidth + 16));
    fseeko(fp, (off_t)e.offset, SEEK_SET);
    const size_t got = fread(raw.data(), 1, raw.size(), fp);
    fclose(fp);
    for (size_t i = 0; i < got && seq.size() < e.len; i++) if (raw[i] != '\n' && raw[i] != '\r') seq.push_back(raw[i]);
    return seq;
}

}  // namespace bamio
