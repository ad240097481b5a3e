// Streaming file pipeline (see stream.hpp).  Stages and the threads that run them:
//
//   reader thread(s)      file -> compressed chunks (BGZF blocks grouped to 8 MB of text, sharing the read buffer) -> inflate
//                         tasks on the pool (fast_inflate.hpp, zlib as fallback);
//                         plain / gzip FASTQ: one zlib stream per file (a gzip stream cannot be split)
//   walker (caller)       byte stream -> records (BAM: block_size chain; single-end: runs of back-to-back records, paired:
//                         mates paired by name; FASTQ: four lines), cut into tasks of at most kSlabReads reads, each with a
//                         slab from the fixed pool
//   pool workers          parse task: fields / tags -> string arenas, bases -> 2-bit words + N mask straight into the
//                         slab's buffers (page-locked in the background, cached across calls), --trim lengths per library;
//                         format task: per-read rows -> text (gzip member for .gz outputs)
//   one thread per GPU    two slabs in flight (slab_api.hpp): H2D, kernels, D2H overlap across slabs
//   committer thread      writes the formatted slabs in input order, merges bulk tables, recycles slabs
//
// Memory is bounded by the slab pool and by the number of inflated chunks in flight, not by the file size.
// 10x mode (nb200_fastq_to_counts): raw R1 / R2 FASTQ; the parse task keeps the pairs fastq-to-bam would correct
// (tenx_select) and the GPU threads correct their barcodes slab by slab (slab_api.hpp: lane_cb_*).
#include "stream.hpp"

#include <zlib.h>

#include <algorithm>
#include <array>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <cstring>
#include <deque>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string_view>
#include <thread>
#include <unordered_map>

#include "fast_inflate.hpp"
#include "ingest.hpp"
#include "library.hpp"
#include "pandas_na.hpp"
#include "slab_api.hpp"
#include "trim.hpp"
#include "umi_code.hpp"

namespace nb200 {
namespace {

constexpr size_t kChunkBytes = 8u << 20;        // inflated bytes per chunk (one inflate task)
constexpr size_t kSlabReads = 1u << 17;         // reads (pairs) per slab at most: one parse task, one GPU batch, one format task per library
constexpr size_t kSlabSeqBytes = kSlabReads * 64;   // packed bytes per mate buffer (64 B stride = reads up to 160 bases)

static bool ends_with_ci(const std::string &s, const char *suf) {
    const size_t n = strlen(suf);
    if (s.size() < n) return false;
    for (size_t i = 0; i < n; i++) if (tolower((unsigned char)s[s.size() - n + i]) != suf[i]) return false;
    return true;
}

// ---- shared failure state -------------------------------------------------------------------------
static double g_wait_block = 0.0, g_wait_slab = 0.0;          // walker-thread waits of the last run (NB200_TRACE)
static std::atomic<uint64_t> g_ns_inflate{0}, g_ns_parse{0}, g_ns_format{0};   // summed over the pool threads
static std::atomic<uint64_t> g_ns_gpu_wait{0}, g_ns_gpu_submit{0}, g_ns_write{0}, g_ns_intern{0};
static inline double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

struct Abort {
    std::atomic<bool> flag{false};
    std::mutex m;
    std::string what;
    bool io = false;
    void set(const std::string &w, bool is_io = false) {
        std::lock_guard<std::mutex> g(m);
        if (!flag.exchange(true)) { what = w; io = is_io; }
    }
};

// ---- worker pool: three priorities, downstream work first (keeps memory bounded) ---------------------------
class Pool {
public:
    enum { FORMAT = 0, PARSE = 1, INFLATE = 2 };
    Pool(int threads, Abort &ab) : ab_(ab) {
        for (int t = 0; t < std::max(1, threads); t++) th_.emplace_back([this] { run(); });
    }
    ~Pool() { stop(); }
    void push(int prio, std::function<void()> fn) {
        { std::lock_guard<std::mutex> g(m_); q_[prio].push_back(std::move(fn)); }
        cv_.notify_one();
    }
    void stop() {
        { std::lock_guard<std::mutex> g(m_); stop_ = true; }
        cv_.notify_all();
        for (auto &t : th_) if (t.joinable()) t.join();
        th_.clear();
    }
private:
    void run() {
        for (;;) {
            std::function<void()> fn;
            {
                std::unique_lock<std::mutex> g(m_);
                cv_.wait(g, [&] { return stop_ || !q_[0].empty() || !q_[1].empty() || !q_[2].empty(); });
                int p = !q_[0].empty() ? 0 : (!q_[1].empty() ? 1 : (!q_[2].empty() ? 2 : -1));
                if (p < 0) return;                      // stop requested and nothing left
                fn = std::move(q_[p].front());
                q_[p].pop_front();
            }
            try { fn(); } catch (const IoError &e) { ab_.set(e.what(), true); } catch (const std::exception &e) { ab_.set(e.what()); }
        }
    }
    Abort &ab_;
    std::mutex m_;
    std::condition_variable cv_;
    std::deque<std::function<void()>> q_[3];
    bool stop_ = false;
    std::vector<std::thread> th_;
};

template <class T>
class Channel {                                  // unbounded MPMC queue with close(); bounded by the slab pool upstream
public:
    void push(T v) { { std::lock_guard<std::mutex> g(m_); q_.push_back(std::move(v)); } cv_.notify_one(); }
    bool pop(T &out) {                           // false: closed and empty
        std::unique_lock<std::mutex> g(m_);
        cv_.wait(g, [&] { return closed_ || !q_.empty(); });
        if (q_.empty()) return false;
        out = std::move(q_.front()); q_.pop_front();
        return true;
    }
    bool try_pop(T &out) {
        std::lock_guard<std::mutex> g(m_);
        if (q_.empty()) return false;
        out = std::move(q_.front()); q_.pop_front();
        return true;
    }
    void close() { { std::lock_guard<std::mutex> g(m_); closed_ = true; } cv_.notify_all(); }
private:
    std::mutex m_;
    std::condition_variable cv_;
    std::deque<T> q_;
    bool closed_ = false;
};

// ---- byte sources -----------------------------------------------------------------------------------
struct Block { std::unique_ptr<char[]> data; size_t n = 0; };
using BlockP = std::shared_ptr<Block>;

class ByteSource {
public:
    virtual ~ByteSource() {}
    virtual BlockP next() = 0;                   // nullptr at end of stream; throws
};

// plain or gzip file through zlib, one stream, one thread ahead of the consumer
class GzSource : public ByteSource {
public:
    GzSource(const std::string &path, Abort &ab) : path_(path), ab_(ab) {
        f_ = gzopen(path.c_str(), "rb");
        if (!f_) throw IoError("cannot open " + path);
        gzbuffer(f_, 1 << 20);
        th_ = std::thread([this] { run(); });
    }
    ~GzSource() override {
        { std::lock_guard<std::mutex> g(m_); quit_ = true; }
        cv_.notify_all();
        if (th_.joinable()) th_.join();
        if (f_) gzclose(f_);
    }
    BlockP next() override {
        std::unique_lock<std::mutex> g(m_);
        cv_.wait(g, [&] { return !q_.empty() || done_ || ab_.flag; });
        if (!err_.empty()) throw IoError(err_);
        if (q_.empty()) return nullptr;
        BlockP b = std::move(q_.front()); q_.pop_front();
        g.unlock();
        cv_.notify_all();
        return b;
    }
private:
    void run() {
        const size_t kBlk = 32u << 20;
        for (;;) {
            {
                std::unique_lock<std::mutex> g(m_);
                cv_.wait(g, [&] { return q_.size() < 4 || quit_ || ab_.flag; });
                if (quit_ || ab_.flag) break;
            }
            auto b = std::make_shared<Block>();
            b->data.reset(new char[kBlk]);
            size_t got = 0;
            while (got < kBlk) {
                const int n = gzread(f_, b->data.get() + got, (unsigned)std::min<size_t>(kBlk - got, 1u << 30));
                if (n < 0) { std::lock_guard<std::mutex> g(m_); err_ = "read error in " + path_; done_ = true; cv_.notify_all(); return; }
                if (n == 0) break;
                got += (size_t)n;
            }
            b->n = got;
            std::lock_guard<std::mutex> g(m_);
            if (got) q_.push_back(std::move(b));
            if (got < kBlk) { done_ = true; cv_.notify_all(); return; }
            cv_.notify_all();
        }
        std::lock_guard<std::mutex> g(m_);
        done_ = true;
        cv_.notify_all();
    }
    std::string path_;
    Abort &ab_;
    gzFile f_ = nullptr;
    std::thread th_;
    std::mutex m_;
    std::condition_variable cv_;
    std::deque<BlockP> q_;
    bool done_ = false, quit_ = false;
    std::string err_;
};

// BGZF (BAM, bgzipped FASTQ): a reader thread groups the compressed blocks into chunks, the pool inflates the chunks
// in parallel, the consumer gets them back in file order
class BgzfSource : public ByteSource {
public:
    static bool is_bgzf(const std::string &path) {
        FILE *f = fopen(path.c_str(), "rb");
        if (!f) throw IoError("cannot open " + path);
        unsigned char h[18];
        const size_t n = fread(h, 1, sizeof h, f);
        fclose(f);
        return n == 18 && h[0] == 31 && h[1] == 139 && (h[3] & 4) && h[12] == 'B' && h[13] == 'C';
    }
    BgzfSource(const std::string &path, Pool &pool, Abort &ab, int max_inflight) : path_(path), pool_(pool), ab_(ab), max_inflight_(std::max(2, max_inflight)) {
        f_ = fopen(path.c_str(), "rb");
        if (!f_) throw IoError("cannot open " + path);
        th_ = std::thread([this] { try { run(); } catch (const std::exception &e) { fail(e.what()); } });
    }
    ~BgzfSource() override {
        quit_ = true;
        { std::lock_guard<std::mutex> g(st_->m); }
        st_->cv.notify_all();
        if (th_.joinable()) th_.join();
        // inflate tasks still queued hold a shared_ptr to the state they touch
        if (f_) fclose(f_);
    }
    BlockP next() override {
        std::unique_lock<std::mutex> g(st_->m);
        st_->cv.wait(g, [&] { return st_->ready.count(next_out_) || (st_->eof && next_out_ >= st_->issued) || !st_->err.empty() || ab_.flag; });
        if (!st_->err.empty()) throw IoError(st_->err);
        auto it = st_->ready.find(next_out_);
        if (it == st_->ready.end()) return nullptr;
        BlockP b = std::move(it->second);
        st_->ready.erase(it);
        next_out_++;
        st_->consumed = next_out_;
        g.unlock();
        st_->cv.notify_all();
        return b;
    }
private:
    struct State {                               // shared with the inflate tasks
        std::mutex m;
        std::condition_variable cv;
        std::map<uint64_t, BlockP> ready;
        uint64_t issued = 0, consumed = 0;
        bool eof = false;
        std::string err;
    };
    struct Piece { size_t off, clen, uoff, ulen; };
    void fail(const std::string &w) { { std::lock_guard<std::mutex> g(st_->m); if (st_->err.empty()) st_->err = w; st_->eof = true; } st_->cv.notify_all(); }
    void dispatch(std::shared_ptr<std::string> raw, std::vector<Piece> pieces, size_t utotal) {
        uint64_t id;
        {
            std::unique_lock<std::mutex> g(st_->m);
            st_->cv.wait(g, [&] { return st_->issued - st_->consumed < (uint64_t)max_inflight_ || quit_ || ab_.flag; });
            if (quit_ || ab_.flag) return;
            id = st_->issued++;
        }
        std::shared_ptr<State> st = st_;
        const std::string path = path_;
        pool_.push(Pool::INFLATE, [st, raw, pieces, utotal, id, path] {
            const double t_in = now_s();
            auto b = std::make_shared<Block>();
            b->data.reset(new char[utotal + 1]);
            b->n = utotal;
            z_stream zs;
            bool bad = false;
            static const bool use_zlib = getenv("NB200_ZLIB_INFLATE") != nullptr;
            for (const Piece &p : pieces) {
                if (!p.ulen) continue;
                // own decoder first (fast_inflate.hpp); zlib for whatever it declines, and for the diagnosis of corrupt input
                if (!use_zlib && fast_inflate((const uint8_t *)raw->data() + p.off, p.clen, (uint8_t *)b->data.get() + p.uoff, p.ulen)) continue;
                memset(&zs, 0, sizeof zs);
                if (inflateInit2(&zs, -15) != Z_OK) { bad = true; break; }
                zs.next_in = (Bytef *)raw->data() + p.off; zs.avail_in = (uInt)p.clen;
                zs.next_out = (Bytef *)(b->data.get() + p.uoff); zs.avail_out = (uInt)p.ulen;
                if (inflate(&zs, Z_FINISH) != Z_STREAM_END) bad = true;
                inflateEnd(&zs);
                if (bad) break;
            }
            g_ns_inflate += (uint64_t)((now_s() - t_in) * 1e9);
            { std::lock_guard<std::mutex> g(st->m); if (bad && st->err.empty()) st->err = "corrupt BGZF block in " + path; st->ready[id] = std::move(b); }
            st->cv.notify_all();
        });
    }
    void run() {
        const size_t kRead = 16u << 20;
        auto raw = std::make_shared<std::string>();
        std::vector<Piece> pieces;
        size_t utotal = 0, pos = 0;                 // pos: parse position inside *raw
        bool file_end = false;
        for (;;) {
            // parse every complete block header + body available in raw[pos..]
            while (raw->size() - pos >= 18) {
                const unsigned char *h = (const unsigned char *)raw->data() + pos;
                if (h[0] != 31 || h[1] != 139 || !(h[3] & 4)) throw IoError("not a BGZF block in " + path_);
                const size_t xlen = h[10] | (h[11] << 8);
                if (raw->size() - pos < 12 + xlen) break;
                size_t bsize = 0, q = 12;
                while (q + 4 <= 12 + xlen) {
                    const size_t slen = h[q + 2] | (h[q + 3] << 8);
                    if (h[q] == 'B' && h[q + 1] == 'C' && slen == 2) bsize = (size_t)(h[q + 4] | (h[q + 5] << 8)) + 1;
                    q += 4 + slen;
                }
                if (!bsize || bsize < 12 + xlen + 8) throw IoError("corrupt BGZF header in " + path_);
                if (raw->size() - pos < bsize) break;
                const unsigned char *t = h + bsize - 4;
                const size_t isize = t[0] | (t[1] << 8) | (t[2] << 16) | ((size_t)t[3] << 24);
                pieces.push_back({pos + 12 + xlen, bsize - 12 - xlen - 8, utotal, isize});
                utotal += isize;
                pos += bsize;
                if (utotal >= kChunkBytes) {
                    // hand the chunk over: the pieces are offsets into the read buffer, which the chunks of one read SHARE
                    // (no copy of the unparsed tail per chunk: that made the reader thread the bottleneck)
                    dispatch(raw, std::move(pieces), utotal);
                    pieces.clear(); utotal = 0;
                }
            }
            if (file_end) break;
            if (quit_ || ab_.flag) return;
            // next read: the blocks parsed so far go out (their offsets belong to this buffer), the partial block at its
            // end (< 64 KB) moves to the front of a new one
            if (!pieces.empty()) { dispatch(raw, std::move(pieces), utotal); pieces.clear(); utotal = 0; }
            {
                auto next_raw = std::make_shared<std::string>();
                next_raw->reserve(raw->size() - pos + kRead);
                next_raw->append(*raw, pos, std::string::npos);
                raw = next_raw; pos = 0;
            }
            const size_t have = raw->size();
            raw->resize(have + kRead);
            const size_t n = fread(&(*raw)[have], 1, kRead, f_);
            raw->resize(have + n);
            if (n == 0) { file_end = true; continue; }
        }
        if (raw->size() != pos) throw IoError("truncated BGZF block at the end of " + path_);
        if (!pieces.empty()) dispatch(raw, std::move(pieces), utotal);
        { std::lock_guard<std::mutex> g(st_->m); st_->eof = true; }
        st_->cv.notify_all();
    }
    std::string path_;
    Pool &pool_;
    Abort &ab_;
    int max_inflight_;
    FILE *f_ = nullptr;
    std::thread th_;
    std::atomic<bool> quit_{false};
    std::shared_ptr<State> st_ = std::make_shared<State>();
    uint64_t next_out_ = 0;
};

// ---- cursor over a byte source: contiguous views, copies only what straddles two blocks --------------------------
struct Keep {                                    // what the records of one task point into
    std::vector<BlockP> blocks;
    std::vector<std::shared_ptr<std::string>> side;
};

class Cursor {
public:
    explicit Cursor(ByteSource *src) : src_(src) {}
    void attach(Keep *k) { keep_ = k; if (cur_ && keep_) keep_->blocks.push_back(cur_); }
    // n contiguous bytes, or nullptr when the stream ends exactly here (n > 0).  Throws when it ends inside.
    const char *need(size_t n, const char *what) {
        if (!fill()) return nullptr;
        if (cur_->n - pos_ >= n) { const char *p = cur_->data.get() + pos_; pos_ += n; return p; }
        auto s = std::make_shared<std::string>();
        s->reserve(n);
        while (s->size() < n) {
            if (!fill()) throw IoError(std::string("truncated ") + what);
            const size_t take = std::min(n - s->size(), cur_->n - pos_);
            s->append(cur_->data.get() + pos_, take);
            pos_ += take;
        }
        keep_->side.push_back(s);
        return s->data();
    }
    // one text line without its terminator; false at end of stream
    bool line(const char *&p, size_t &len) {
        if (!fill()) return false;
        const char *b = cur_->data.get() + pos_;
        const char *nl = (const char *)memchr(b, '\n', cur_->n - pos_);
        if (nl) {
            p = b; len = (size_t)(nl - b); pos_ += len + 1;
        } else {
            auto s = std::make_shared<std::string>(b, cur_->n - pos_);
            pos_ = cur_->n;
            for (;;) {
                if (!fill()) break;                 // last line without a newline
                const char *c = cur_->data.get() + pos_;
                const char *e = (const char *)memchr(c, '\n', cur_->n - pos_);
                if (e) { s->append(c, (size_t)(e - c)); pos_ += (size_t)(e - c) + 1; break; }
                s->append(c, cur_->n - pos_);
                pos_ = cur_->n;
            }
            keep_->side.push_back(s);
            p = s->data(); len = s->size();
        }
        while (len && (p[len - 1] == '\r')) len--;
        return true;
    }
private:
    bool fill() {                                // a current block with unread bytes, or false at the end
        while (!cur_ || pos_ >= cur_->n) {
            if (end_) return false;
            const double t0 = now_s();
            cur_ = src_->next();
            g_wait_block += now_s() - t0;
            pos_ = 0;
            if (!cur_) { end_ = true; return false; }
            if (keep_) keep_->blocks.push_back(cur_);
        }
        return true;
    }
    ByteSource *src_;
    Keep *keep_ = nullptr;
    BlockP cur_;
    size_t pos_ = 0;
    bool end_ = false;
};

// ---- slabs --------------------------------------------------------------------------------------------
struct StrCol {                                  // strings back to back
    std::string data;
    std::vector<uint32_t> off;
    void reset(size_t n) { data.clear(); off.assign(1, 0); off.reserve(n + 1); }
    void add(const char *p, size_t n) { data.append(p, n); off.push_back((uint32_t)data.size()); }
    const char *ptr(size_t i) const { return data.data() + off[i]; }
    size_t len(size_t i) const { return off[i + 1] - off[i]; }
};

struct Slab {
    // packed reads in, per-read results out.  Page-aligned plain memory that a background thread page-locks while the
    // slab is idle (cudaHostRegister): the first slabs of a run go through the driver's staging copies, the later ones
    // (and every slab of a later call in the same process: the pool is cached) are true asynchronous DMA targets.
    uint8_t *p1 = nullptr, *p2 = nullptr;
    uint16_t *l1 = nullptr, *l2 = nullptr;
    std::vector<nb200_read_result *> res;
    std::vector<int32_t *> feats;
    std::vector<uint16_t *> lt1, lt2;              // --trim: per library, bases kept of every read / mate (else empty)
    struct Buf { void *p; size_t bytes; bool pinned, tried; };
    std::vector<Buf> bufs;
    void *grab(size_t bytes) {
        void *p = nullptr;
        bytes = (bytes + 4095) & ~(size_t)4095;
        if (posix_memalign(&p, 4096, bytes) != 0 || !p) throw std::runtime_error("out of host memory for the read slabs");
        bufs.push_back(Buf{p, bytes, false, false});
        return p;
    }
    bool all_pinned() const { for (const Buf &b : bufs) if (!b.tried) return false; return true; }     // (or given up on)
    void release() {
        for (Buf &b : bufs) { if (b.pinned) lane_unpin(b.p); free(b.p); }
        bufs.clear();
    }
    // one use
    uint64_t seq = 0;
    size_t n = 0;
    bool paired = false, has_tags = false;
    nb200_reads r1{}, r2{};
    StrCol names, cb, ub, ur, gn;
    std::vector<int64_t> pos1, pos2;
    std::vector<std::string> out;                                        // per library: rows (a gzip member for .gz)
    std::vector<std::unordered_map<std::string, uint64_t>> bulk;         // per library, untagged input: id list -> reads
    uint64_t bases1 = 0, bases2 = 0, called = 0;
    uint64_t *key = nullptr;                                             // counts mode: cell << 32 | umi per read
    uint64_t tagged = 0;                                                 // counts mode: reads with a CB or UB value
    // 10x mode: raw cell barcodes and their phred values (n x cb_len) of the pairs in the slab; fastq-to-bam's counters
    uint8_t *cbc = nullptr, *cbq = nullptr;
    uint64_t pairs = 0, name_mismatch = 0, too_short = 0, no_remaining_seq = 0;
    uint64_t cbn[6] = {0, 0, 0, 0, 0, 0};                                // lane_cb_counters
};

// ---- counts mode: CB / UB strings -> key = cell << 32 | umi -------------------------------------------------------
// Cells: one dictionary for the call, shared by every context (ids agree across GPUs), ids in first-seen order; the
// ranks by CB bytes are computed once at the end (lane_rows_count).  UMIs: only equality matters (report groups rows by
// it, nimble/__main__.py:254-293): an ACGTN string of up to 13 bases is its bijective base-5 value (< 2^31, injective
// across lengths, no dictionary), anything else is interned with bit 31 set.  A pool thread looks a CB up in a map of
// its own first (CellCache) and takes a shard's lock only for the CB's first sight on that thread.
class BarcodeDict {
public:
    BarcodeDict() { static std::atomic<uint64_t> calls{0}; gen_ = ++calls; }
    uint64_t gen() const { return gen_; }        // tells the per-thread caches of one call from those of another
    uint32_t cell(std::string_view s) { return get(cells_, n_cells_, s); }
    uint32_t umi(std::string_view s) { return get(umis_, n_umis_, s) | kUmiInterned; }
    std::vector<std::string> cell_names() const {                        // id -> CB
        std::vector<std::string> v(n_cells_.load());
        for (const Shard &S : cells_) for (const auto &kv : S.map) v[kv.second] = kv.first;
        return v;
    }
private:
    static constexpr size_t kShards = 64;
    struct Shard { std::mutex m; std::unordered_map<std::string, uint32_t> map; };
    static uint32_t get(Shard *sh, std::atomic<uint32_t> &ctr, std::string_view s) {
        Shard &S = sh[std::hash<std::string_view>()(s) % kShards];
        std::lock_guard<std::mutex> g(S.m);
        std::string k(s);
        auto it = S.map.find(k);
        if (it != S.map.end()) return it->second;
        const uint32_t id = ctr++;
        if (id >= 0x7FFFFFFFu) throw LimitError("more than 2^31 distinct cell barcodes or UMIs");
        S.map.emplace(std::move(k), id);
        return id;
    }
    Shard cells_[kShards], umis_[kShards];
    std::atomic<uint32_t> n_cells_{0}, n_umis_{0};
    uint64_t gen_ = 0;
};

// CB -> cell id for one pool thread, kept across the slabs of a call: a slab holds most cells of a large sample once,
// so a per-slab map sends nearly every read to the shared dictionary (its lock, a string copy); a thread's own map
// stops doing so after its first slabs.  Bounded: beyond kMax cells the rest go to the shared dictionary.
struct CellCache {
    static constexpr size_t kMax = 1u << 18;
    uint64_t gen = 0;
    std::unordered_map<size_t, std::pair<uint32_t, std::string>> ids;      // hash of the CB -> (id, CB)
};

// the key's low half for a UMI that is not a pandas NA token (seen: the slab's interned UMIs, saves the shared lock)
static inline uint32_t umi_id(std::string_view ub, BarcodeDict &bc, std::unordered_map<std::string_view, uint32_t> &seen) {
    uint32_t u;
    if (umi_code(ub, u)) return u;
    auto v = seen.find(ub);
    if (v == seen.end()) v = seen.emplace(ub, bc.umi(ub)).first;
    return v->second;
}

// keys of a parsed slab (runs on the pool, inside the parse task): invalid barcodes (absent, empty, a pandas NA token:
// `report` drops those rows, nimble/__main__.py:244-245) -> NB200_NO_BARCODE
static void slab_keys(Slab &S, BarcodeDict &bc) {
    const double t_in = now_s();
    static thread_local CellCache cc;
    if (cc.gen != bc.gen()) { cc.ids.clear(); cc.gen = bc.gen(); }
    std::unordered_map<std::string_view, uint32_t> umis;
    S.tagged = 0;
    for (size_t i = 0; i < S.n; i++) {
        const std::string_view cb(S.cb.ptr(i), S.cb.len(i)), ub(S.ub.ptr(i), S.ub.len(i));
        S.tagged += !cb.empty() || !ub.empty();
        if (pandas_na(cb) || pandas_na(ub)) { S.key[i] = NB200_NO_BARCODE; continue; }
        const size_t h = std::hash<std::string_view>()(cb);
        auto c = cc.ids.find(h);
        uint32_t cid;
        if (c != cc.ids.end() && c->second.second == cb) cid = c->second.first;
        else {
            cid = bc.cell(cb);
            if (c == cc.ids.end() && cc.ids.size() < CellCache::kMax) cc.ids.emplace(h, std::make_pair(cid, std::string(cb)));
        }
        S.key[i] = ((uint64_t)cid << 32) | umi_id(ub, bc, umis);
    }
    g_ns_intern += (uint64_t)((now_s() - t_in) * 1e9);
}

struct Entry {                                   // one read (pair) as the walker found it
    const char *a = nullptr, *b = nullptr;       // BAM: record bodies of mate 1 / mate 2; FASTQ: the two sequences
    uint32_t la = 0, lb = 0;
    const char *name = nullptr;                  // FASTQ only
    uint32_t ln = 0;
    const char *qa = nullptr, *qb = nullptr;     // FASTQ only: quality lines (phred + 33) of the two mates, when --trim wants them
    const char *name2 = nullptr;                 // 10x mode: R2's name (process_pair compares the two)
    uint32_t ln2 = 0;
};

struct Task {
    bool bam = false, paired = false;
    std::vector<Entry> e;
    Keep keep;
    uint32_t max1 = 1, max2 = 1;                 // longest read per mate
    // single-end BAM: runs of records that lie back to back in memory (p = block_size field of the first one); the
    // walker only chains through the sizes, the parse task walks the runs again and does the rest in parallel
    struct Seg { const char *p; uint32_t n; };
    std::vector<Seg> segs;
    size_t n_seg_records = 0, seg_bytes_of_last = 0;    // (bytes of the last run so far: the next record extends it when it starts right there)
    Slab *slab = nullptr;
    const std::vector<TrimTable> *trims = nullptr;   // per library (--trim), or nullptr
    BarcodeDict *bc = nullptr;                   // counts mode
    int cb_len = 0, umi_len = 0;                 // 10x mode when cb_len > 0 (tenx_select)
    std::string qconv;                           // 10x mode with --trim: the qualities as fastq-to-bam's BAM stores them
};

static inline uint32_t le32(const unsigned char *p) { return p[0] | (p[1] << 8) | (p[2] << 16) | ((uint32_t)p[3] << 24); }
static inline uint32_t stride_for(uint32_t max_len) { const uint32_t w = std::max(1u, (max_len + 31) / 32); return (12 * w + 15) & ~15u; }

// ---- packing ---------------------------------------------------------------------------------------------
// codes[i] in 0..3, or 4 for anything that is not A C G T: -> [seq u64 x words][N mask u32 x words], zero padded
static void pack_codes(const uint8_t *codes, uint32_t L, uint8_t *rec, uint32_t words, uint32_t stride) {
    uint64_t *seq = reinterpret_cast<uint64_t *>(rec);
    uint32_t *nm = reinterpret_cast<uint32_t *>(rec + (size_t)words * 8);
    uint32_t j = 0;
    for (uint32_t w = 0; w < words; w++) {
        uint64_t acc = 0;
        uint32_t nacc = 0;
        const uint32_t e = std::min(L, j + 32);
        for (int sh = 0; j < e; j++, sh++) {
            const uint32_t v = codes[j];
            acc |= (uint64_t)(v & 3u) << (2 * sh);
            nacc |= (v >> 2) << sh;
        }
        seq[w] = acc; nm[w] = nacc;
    }
    for (size_t t = (size_t)words * 12; t < stride; t++) rec[t] = 0;
}

struct Luts {
    uint8_t ascii[256];          // base letter -> 0..3 / 4
    uint8_t nib[16];             // BAM 4-bit code -> 0..3 / 4
    uint8_t pair[256];           // BAM byte (high nibble = first base): bits 0-3 two 2-bit codes, bits 4-5 their N flags
    Luts() {
        memset(ascii, 4, sizeof ascii);
        ascii['A'] = ascii['a'] = 0; ascii['C'] = ascii['c'] = 1; ascii['G'] = ascii['g'] = 2; ascii['T'] = ascii['t'] = 3;
        memset(nib, 4, sizeof nib);
        nib[1] = 0; nib[2] = 1; nib[4] = 2; nib[8] = 3;     // =ACMGRSVTWYHKDBN
        for (int v = 0; v < 256; v++) {
            const uint8_t a = nib[v >> 4], b = nib[v & 15];
            pair[v] = (uint8_t)((a & 3) | ((b & 3) << 2) | ((a >> 2) << 4) | ((b >> 2) << 5));
        }
    }
};
static const Luts &luts() { static const Luts l; return l; }

struct BamView {                                  // fields of one BAM record body
    const unsigned char *name = nullptr, *seq = nullptr, *qual = nullptr;
    const char *tag[4] = {nullptr, nullptr, nullptr, nullptr};   // CB UB UR GN (Z)
    uint32_t name_len = 0, l_seq = 0, tag_len[4] = {0, 0, 0, 0}, flag = 0;
    int64_t pos = -1;
};

static void bam_fields(const char *body, uint32_t size, BamView &x, bool want_tags) {
    const unsigned char *r = (const unsigned char *)body, *end = r + size;
    if (size < 32) throw std::runtime_error("truncated BAM record");
    x.pos = (int64_t)(int32_t)le32(r + 4) + 1;
    const uint32_t l_name = r[8];
    const uint32_t n_cigar = r[12] | (r[13] << 8);
    x.flag = r[14] | (r[15] << 8);
    x.l_seq = le32(r + 16);
    const unsigned char *q = r + 32;
    x.name = q; x.name_len = l_name ? l_name - 1 : 0;
    q += l_name + 4 * (size_t)n_cigar;
    x.seq = q;
    x.qual = q + (x.l_seq + 1) / 2;
    q += (x.l_seq + 1) / 2 + (size_t)x.l_seq;
    if (q > end) throw std::runtime_error("corrupt BAM record");
    if (!want_tags) return;
    while (q + 3 <= end) {
        const char t0 = (char)q[0], t1 = (char)q[1], ty = (char)q[2]; q += 3;
        size_t adv = 0;
        const char *zs = nullptr;
        switch (ty) {
        case 'Z': case 'H': { zs = (const char *)q; adv = strnlen(zs, end - q) + 1; break; }
        case 'A': case 'c': case 'C': adv = 1; break;
        case 's': case 'S': adv = 2; break;
        case 'i': case 'I': case 'f': adv = 4; break;
        case 'B': { if (q + 5 > end) throw std::runtime_error("corrupt BAM tag");
                    const char sub = (char)q[0]; const uint32_t cnt = le32(q + 1);
                    const int es = (sub == 'c' || sub == 'C') ? 1 : (sub == 's' || sub == 'S') ? 2 : 4; adv = 5 + (size_t)cnt * es; break; }
        default: throw std::runtime_error("unknown BAM tag type");
        }
        if (zs) {
            int slot = -1;
            if (t0 == 'C' && t1 == 'B') slot = 0; else if (t0 == 'U' && t1 == 'B') slot = 1;
            else if (t0 == 'U' && t1 == 'R') slot = 2; else if (t0 == 'G' && t1 == 'N') slot = 3;
            if (slot >= 0) { x.tag[slot] = zs; x.tag_len[slot] = (uint32_t)(adv - 1); }
        }
        q += adv;
    }
}

static void pack_bam(const BamView &x, uint8_t *rec, uint32_t words, uint32_t stride) {
    const Luts &lt = luts();
    const uint32_t L = x.l_seq;
    if (!(x.flag & 0x10)) {
        // forward: one table lookup per BYTE (two bases): 4 bits of 2-bit codes + 2 N flags
        uint64_t *seq = reinterpret_cast<uint64_t *>(rec);
        uint32_t *nm = reinterpret_cast<uint32_t *>(rec + (size_t)words * 8);
        const uint32_t nbytes = (L + 1) / 2;
        uint32_t j = 0;
        for (uint32_t w = 0; w < words; w++) {
            uint64_t acc = 0;
            uint32_t nacc = 0;
            const uint32_t e = std::min(nbytes, j + 16);
            for (int sh = 0; j < e; j++, sh++) {
                const uint32_t v = lt.pair[x.seq[j]];
                acc |= (uint64_t)(v & 15u) << (4 * sh);
                nacc |= (v >> 4) << (2 * sh);
            }
            seq[w] = acc; nm[w] = nacc;
        }
        if (L & 1) {                               // the low nibble of the last byte is padding, not a base
            const uint32_t w = (L - 1) >> 5, b = L & 31;      // base L sits at bit b of word (L >> 5) == w unless b == 0
            if (b) { seq[w] &= (1ull << (2 * b)) - 1; nm[w] &= (1u << b) - 1; }
        }
        for (size_t t = (size_t)words * 12; t < stride; t++) rec[t] = 0;
        return;
    }
    uint8_t codes[NB200_MAX_READ_LEN + 2];
    for (uint32_t i = 0; i + 1 < L; i += 2) { const unsigned v = x.seq[i >> 1]; codes[i] = lt.nib[v >> 4]; codes[i + 1] = lt.nib[v & 15]; }
    if (L & 1) codes[L - 1] = lt.nib[x.seq[L >> 1] >> 4];
    std::reverse(codes, codes + L);                // stored reverse-complemented: restore the read as sequenced
    for (uint32_t i = 0; i < L; i++) if (codes[i] < 4) codes[i] = 3 - codes[i];
    pack_codes(codes, L, rec, words, stride);
}
static void pack_ascii(const char *s, uint32_t L, uint8_t *rec, uint32_t words, uint32_t stride) {
    uint8_t codes[NB200_MAX_READ_LEN + 2];
    const Luts &lt = luts();
    for (uint32_t i = 0; i < L; i++) codes[i] = lt.ascii[(unsigned char)s[i]];
    pack_codes(codes, L, rec, words, stride);
}

// 10x mode, first step of the parse task: keep the pairs fastq-to-bam would hand to the barcode correction
// (process_pair's rules, slice_barcodes) and turn each into what that BAM's records hold: raw CB + phred values into the
// slab, the UMI into the key's low half, read 1 = R1 after barcode and UMI, read 2 = R2.  The rest is counted.
static void tenx_select(Task &t) {
    Slab &S = *t.slab;
    const uint32_t L = (uint32_t)t.cb_len, U = (uint32_t)t.umi_len, bl = L + U;
    const bool want_q = t.trims && !S.lt1.empty();
    std::unordered_map<std::string_view, uint32_t> umis;
    if (want_q) {
        size_t bytes = 0;
        for (const Entry &e : t.e) bytes += e.la + e.lb;
        t.qconv.clear();
        t.qconv.reserve(bytes);                       // (no reallocation below: the entries point into it)
    }
    // the BAM stores phred values (quality byte - 33); align reads 0xFF in the first one as "no qualities"
    auto bam_qual = [&](const char *q, uint32_t n) -> const char * {
        const size_t at = t.qconv.size();
        for (uint32_t j = 0; j < n; j++) t.qconv.push_back((char)(uint8_t)(q[j] - 33));
        return (n && (uint8_t)t.qconv[at] == 0xFF) ? nullptr : t.qconv.data() + at;
    };
    S.pairs = t.e.size(); S.name_mismatch = S.too_short = S.no_remaining_seq = 0;
    size_t o = 0;
    for (size_t i = 0; i < t.e.size(); i++) {
        Entry e = t.e[i];
        if (!name_eq_stripped(e.name, e.ln, e.name2, e.ln2)) { S.name_mismatch++; continue; }
        if (e.la < bl) { S.too_short++; continue; }
        if (e.la == bl) { S.no_remaining_seq++; continue; }
        // what writing the BAM (a name over 254 bytes) or aligning it (a read over 500 bases) refuses: the two steps fail
        // only when the pair is written, i.e. its barcode gets a correction, so the device decides (cb_key_kernel).  The
        // pair still takes part in the correction and its cache rule; an over-long read goes to the kernels empty.
        uint32_t nl = e.ln;
        if (nl >= 2 && e.name[nl - 2] == '/' && e.name[nl - 1] == '1') nl -= 2;
        const uint64_t flags = (nl > 254 ? kTenxLongName : 0) | ((e.la - bl > NB200_MAX_READ_LEN || e.lb > NB200_MAX_READ_LEN) ? kTenxLongRead : 0);
        memcpy(S.cbc + o * L, e.a, L);
        for (uint32_t j = 0; j < L; j++) S.cbq[o * L + j] = (uint8_t)(e.qa[j] - 33);
        const std::string_view umi(e.a + L, U);
        S.key[o] = (flags << 32) | (pandas_na(umi) ? kTenxNaUmi : umi_id(umi, *t.bc, umis));
        if (want_q) { e.qa = bam_qual(e.qa + bl, e.la - bl); e.qb = bam_qual(e.qb, e.lb); }
        e.a += bl; e.la -= bl;
        if (flags & kTenxLongRead) { e.la = 0; e.lb = 0; }
        t.e[o++] = e;
    }
    t.e.resize(o);
}

// task -> slab (runs on the pool)
static void parse_task(Task &t) {
    if (t.cb_len) tenx_select(t);
    Slab &S = *t.slab;
    const size_t n = t.segs.empty() ? t.e.size() : t.n_seg_records;
    S.n = n; S.paired = t.paired; S.has_tags = t.bam;
    uint32_t w1 = std::max(1u, (t.max1 + 31) / 32), s1 = stride_for(t.max1), w2 = std::max(1u, (t.max2 + 31) / 32), s2 = stride_for(t.max2);
    S.r1 = nb200_reads{S.p1, S.l1, n, s1, w1};
    S.r2 = nb200_reads{S.p2, S.l2, n, s2, w2};
    S.names.reset(n); S.cb.reset(n); S.ub.reset(n); S.ur.reset(n); S.gn.reset(n);
    S.pos1.assign(n, -1); S.pos2.assign(n, -1);
    S.bases1 = S.bases2 = 0;
    const bool trimming = t.trims && !S.lt1.empty();
    // --trim: bases kept per library (the packed record holds the whole read; every library's kernels get their own lengths)
    auto trimmed = [&](std::vector<uint16_t *> &lt, size_t i, uint32_t L, const uint8_t *qual, int offset, bool reversed) {
        for (size_t li = 0; li < lt.size(); li++) {
            const TrimTable &T = (*t.trims)[li];
            lt[li][i] = (uint16_t)((T.on && qual && L) ? T.keep(qual, L, offset, reversed) : L);
        }
    };
    size_t seg_i = 0, seg_left = t.segs.empty() ? 0 : t.segs[0].n;
    const char *seg_p = t.segs.empty() ? nullptr : t.segs[0].p;
    for (size_t i = 0; i < n; i++) {
        Entry seg_e;
        if (!t.segs.empty()) {                       // next record of the current run
            while (seg_left == 0) { seg_i++; seg_left = t.segs[seg_i].n; seg_p = t.segs[seg_i].p; }
            const uint32_t size = le32((const unsigned char *)seg_p);
            seg_e.a = seg_p + 4; seg_e.la = size;
            seg_p += 4 + (size_t)size; seg_left--;
        }
        const Entry &e = t.segs.empty() ? t.e[i] : seg_e;
        if (trimming && !t.bam) {
            const int off = t.cb_len ? 0 : 33;         // 10x mode: phred values already (tenx_select)
            trimmed(S.lt1, i, e.la, (const uint8_t *)e.qa, off, false);
            if (t.paired) trimmed(S.lt2, i, e.lb, (const uint8_t *)e.qb, off, false);
        }
        if (t.bam) {
            BamView a, b;
            if (e.a) bam_fields(e.a, e.la, a, true);
            if (e.b) bam_fields(e.b, e.lb, b, false);
            if (trimming) {                          // (bam_fields has checked that the quality bytes lie inside the record)
                auto one = [&](const char *body, const BamView &v, std::vector<uint16_t *> &lt) {
                    const bool has_q = body && v.l_seq && v.qual[0] != 0xFF;                          // 0xFF: qualities absent
                    trimmed(lt, i, body ? v.l_seq : 0, has_q ? v.qual : nullptr, 0, (v.flag & 0x10) != 0);
                };
                one(e.a, a, S.lt1);
                if (t.paired) one(e.b, b, S.lt2);
            }
            const BamView &nm = e.a ? a : b;
            S.names.add((const char *)nm.name, nm.name_len);
            if (e.a) {
                pack_bam(a, S.p1 + i * (size_t)s1, w1, s1); S.l1[i] = (uint16_t)a.l_seq; S.bases1 += a.l_seq;
                S.cb.add(a.tag[0], a.tag_len[0]); S.ub.add(a.tag[1], a.tag_len[1]); S.ur.add(a.tag[2], a.tag_len[2]); S.gn.add(a.tag[3], a.tag_len[3]);
                S.pos1[i] = a.pos;
            } else {
                memset(S.p1 + i * (size_t)s1, 0, s1); S.l1[i] = 0;
                S.cb.add("", 0); S.ub.add("", 0); S.ur.add("", 0); S.gn.add("", 0);
            }
            if (t.paired) {
                if (e.b) { pack_bam(b, S.p2 + i * (size_t)s2, w2, s2); S.l2[i] = (uint16_t)b.l_seq; S.bases2 += b.l_seq; S.pos2[i] = b.pos; }
                else { memset(S.p2 + i * (size_t)s2, 0, s2); S.l2[i] = 0; }
            }
        } else {
            S.names.add(e.name, e.ln);
            pack_ascii(e.a, e.la, S.p1 + i * (size_t)s1, w1, s1); S.l1[i] = (uint16_t)e.la; S.bases1 += e.la;
            if (t.paired) { pack_ascii(e.b, e.lb, S.p2 + i * (size_t)s2, w2, s2); S.l2[i] = (uint16_t)e.lb; S.bases2 += e.lb; }
        }
    }
    if (t.bc && !t.cb_len) slab_keys(S, *t.bc);
}

// ---- output ----------------------------------------------------------------------------------------------
static void gzip_member(const std::string &in, std::string &out) {       // members concatenate into one valid .gz file
    z_stream zs;
    memset(&zs, 0, sizeof zs);
    if (deflateInit2(&zs, 4, Z_DEFLATED, 15 + 16, 8, Z_DEFAULT_STRATEGY) != Z_OK) throw std::runtime_error("deflateInit2 failed");
    out.resize(deflateBound(&zs, (uLong)in.size()) + 64);
    zs.next_in = (Bytef *)in.data(); zs.avail_in = (uInt)in.size();
    zs.next_out = (Bytef *)&out[0]; zs.avail_out = (uInt)out.size();
    const int rc = deflate(&zs, Z_FINISH);
    const size_t n = zs.total_out;
    deflateEnd(&zs);
    if (rc != Z_STREAM_END) throw std::runtime_error("deflate failed");
    out.resize(n);
}

static const char kPerReadHeader[] =
    "nimble_features\tnimble_score\tr1_forward_score\tr1_reverse_score\tr2_forward_score\tr2_reverse_score\t"
    "r1_QNAME\tr1_CB\tr1_UB\tr1_UR\tr1_GN\tr1_POS\tr2_POS\n";

struct LibOut {
    int32_t lib_id = 0;
    int max_hits = 0;
    bool gz = false;
    std::string path, tmp;
    FILE *f = nullptr;
    std::vector<std::pair<const char *, uint32_t>> names;      // feature id -> name
    std::unordered_map<std::string, uint64_t> bulk;
};

static inline void put_uint(std::string &o, uint64_t v) {
    char b[24]; int n = 0;
    do { b[n++] = (char)('0' + v % 10); v /= 10; } while (v);
    while (n) o.push_back(b[--n]);
}

// rows of one slab for one library (runs on the pool)
static void format_slab(Slab &S, size_t li, const LibOut &lo) {
    const size_t n = S.n;
    const nb200_read_result *res = S.res[li];
    const int32_t *feats = S.feats[li];
    const int mh = lo.max_hits;
    std::string text;
    if (S.has_tags) {
        text.reserve(n * 48);
        for (size_t i = 0; i < n; i++) {
            if (!res[i].n_feat) continue;
            S.called += li == 0;
            for (int j = 0; j < res[i].n_feat; j++) {
                if (j) text += ',';
                const auto &nm = lo.names[(size_t)feats[i * (size_t)mh + j]];
                text.append(nm.first, nm.second);
            }
            text += "\t1";
            for (int o = 0; o < 4; o++) { text += '\t'; put_uint(text, res[i].score[o]); }
            text += '\t'; text.append(S.names.ptr(i), S.names.len(i));
            text += '\t'; text.append(S.cb.ptr(i), S.cb.len(i));
            text += '\t'; text.append(S.ub.ptr(i), S.ub.len(i));
            text += '\t'; text.append(S.ur.ptr(i), S.ur.len(i));
            text += '\t'; text.append(S.gn.ptr(i), S.gn.len(i));
            text += '\t'; if (S.pos1[i] > 0) put_uint(text, (uint64_t)S.pos1[i]);
            text += '\t'; if (S.pos2[i] > 0) put_uint(text, (uint64_t)S.pos2[i]);
            text += '\n';
        }
        if (lo.gz && !text.empty()) gzip_member(text, S.out[li]); else S.out[li].swap(text);
    } else {
        auto &m = S.bulk[li];
        m.clear();
        std::string key;
        for (size_t i = 0; i < n; i++) {
            if (!res[i].n_feat) continue;
            S.called += li == 0;
            key.assign((const char *)(feats + i * (size_t)mh), (size_t)res[i].n_feat * 4);
            m[key]++;
        }
    }
}

// ---- the pipeline -----------------------------------------------------------------------------------------
struct SlabCache {                               // idle slabs between calls (never torn down at exit: the CUDA runtime may be gone)
    std::mutex m;
    std::vector<std::unique_ptr<Slab>> slabs;
    std::vector<int> geom;                       // max_hits per library the result buffers were sized for
};
static SlabCache &g_slab_cache = *new SlabCache;

struct Pipeline {
    const FileJob &job;
    Abort ab;
    std::unique_ptr<Pool> pool;
    std::vector<LibOut> libs;
    std::vector<std::unique_ptr<Slab>> slabs;
    Channel<Slab *> free_slabs, to_gpu, to_commit;
    std::vector<std::thread> gpu_threads;
    std::thread committer;
    FileStats stats;
    bool dry = false;
    bool per_read = true;                          // per-read TSVs are written
    bool counts = false;                           // counts TSVs: keys per read, rows kept on the devices
    bool tenx = false;                             // raw 10x R1 / R2 in, cell barcodes corrected on the devices (FileJob)
    BarcodeDict bc;
    std::mutex seg_m;
    std::vector<std::vector<RowSeg>> segs;         // counts mode, per library: the segments of every slab on every context
    uint64_t tagged = 0;

    explicit Pipeline(const FileJob &j) : job(j) {}

    // The slab pool outlives the call (g_slab_cache): page-locking is slow (hundreds of MB/s on some hosts) and is paid
    // once per process, off the critical path, by the pinner thread.
    std::thread pinner;
    std::atomic<bool> stop_pin{false};
    Slab *alloc_slab() {
        const size_t n_libs = dry ? 0 : job.lib_ids.size();
        auto S = std::make_unique<Slab>();
        S->p1 = (uint8_t *)S->grab(kSlabSeqBytes + 256); S->l1 = (uint16_t *)S->grab(kSlabReads * 2 + 64);
        for (size_t li = 0; li < (per_read ? n_libs : 0); li++) {       // (counts only: the per-read results stay on the device)
            S->res.push_back((nb200_read_result *)S->grab(kSlabReads * sizeof(nb200_read_result) + 64));
            S->feats.push_back((int32_t *)S->grab(kSlabReads * (size_t)libs[li].max_hits * 4 + 64));
        }
        if (counts) S->key = (uint64_t *)S->grab(kSlabReads * 8 + 64);
        if (tenx) { S->cbc = (uint8_t *)S->grab(kSlabReads * (size_t)job.cb_len + 64); S->cbq = (uint8_t *)S->grab(kSlabReads * (size_t)job.cb_len + 64); }
        if (!trims.empty())
            for (size_t li = 0; li < n_libs; li++) S->lt1.push_back((uint16_t *)S->grab(kSlabReads * 2 + 64));
        S->out.resize(n_libs); S->bulk.resize(n_libs);
        Slab *raw = S.get();
        slabs.push_back(std::move(S));
        return raw;
    }
    std::atomic<int> to_pin{0};                    // slabs with a buffer the pinner has not seen yet
    void need_mate2(Slab *S) {                     // walker thread, first paired use of the slab
        if (S->p2) return;
        if (S->all_pinned()) to_pin++;
        S->p2 = (uint8_t *)S->grab(kSlabSeqBytes + 256); S->l2 = (uint16_t *)S->grab(kSlabReads * 2 + 64);
        for (size_t li = 0; li < S->lt1.size(); li++) S->lt2.push_back((uint16_t *)S->grab(kSlabReads * 2 + 64));
    }
    std::vector<TrimTable> trims;                  // per library; empty = no --trim anywhere
    std::vector<int> geometry() const {
        std::vector<int> g;
        if (!dry) for (const LibOut &lo : libs) g.push_back(lo.max_hits);
        g.push_back(trims.empty() ? 0 : 1);
        g.push_back((per_read ? 1 : 0) | (counts ? 2 : 0));
        g.push_back(tenx ? job.cb_len : 0);
        return g;
    }
    void start_pool(size_t count, nb200_ctx *bind) {
        {   // slabs of an earlier call in this process, if they have the same shape
            std::lock_guard<std::mutex> g(g_slab_cache.m);
            if (g_slab_cache.geom == geometry() && !g_slab_cache.slabs.empty()) slabs.swap(g_slab_cache.slabs);
            else { for (auto &S : g_slab_cache.slabs) S->release(); g_slab_cache.slabs.clear(); }
        }
        while (slabs.size() > count) { slabs.back()->release(); slabs.pop_back(); }
        for (auto &S : slabs) { S->out.assign(S->out.size(), std::string()); S->called = 0; }
        while (slabs.size() < count) alloc_slab();
        for (auto &S : slabs) { free_slabs.push(S.get()); if (!S->all_pinned()) to_pin++; }
        if (!bind || getenv("NB200_NO_PIN")) return;
        pinner = std::thread([this, bind] {
            try {
                lane_bind_thread(bind);
                while (!stop_pin && !ab.flag) {
                    if (to_pin == 0) { std::this_thread::sleep_for(std::chrono::milliseconds(2)); continue; }   // (paired input may add mate-2 buffers later)
                    Slab *S = nullptr;
                    if (!free_slabs.try_pop(S)) { std::this_thread::sleep_for(std::chrono::milliseconds(1)); continue; }
                    if (S->all_pinned()) { free_slabs.push(S); std::this_thread::sleep_for(std::chrono::microseconds(200)); continue; }
                    for (Slab::Buf &b : S->bufs) if (!b.tried) { b.pinned = lane_pin(b.p, b.bytes); b.tried = true; }
                    to_pin--;
                    free_slabs.push(S);
                }
            } catch (const std::exception &e) { ab.set(e.what()); }
        });
    }
    void stop_pinner() { stop_pin = true; if (pinner.joinable()) pinner.join(); }
    void free_all() {                              // back to the cache (bounded), the rest is released
        std::lock_guard<std::mutex> g(g_slab_cache.m);
        for (auto &S : g_slab_cache.slabs) S->release();
        g_slab_cache.slabs.clear();
        if (getenv("NB200_NO_SLAB_CACHE")) { for (auto &S : slabs) S->release(); slabs.clear(); return; }
        g_slab_cache.geom = geometry();
        g_slab_cache.slabs.swap(slabs);
    }

    // a parsed slab goes to a GPU (or straight to the committer in a dry run)
    void after_parse(Slab *S) { if (dry) to_commit.push(S); else to_gpu.push(S); }
    // a slab with results: format every library's rows on the pool, then commit
    void after_gpu(Slab *S) {
        if (!per_read) { to_commit.push(S); return; }
        auto left = std::make_shared<std::atomic<size_t>>(libs.size());
        for (size_t li = 0; li < libs.size(); li++)
            pool->push(Pool::FORMAT, [this, S, li, left] {
                const double t_in = now_s();
                try { if (!ab.flag) format_slab(*S, li, libs[li]); } catch (const std::exception &e) { ab.set(e.what()); }
                g_ns_format += (uint64_t)((now_s() - t_in) * 1e9);
                if (left->fetch_sub(1) == 1) to_commit.push(S);
            });
    }

    void gpu_main(nb200_ctx *c, int ctx_index) {
        Slab *fly[kFileLanes] = {nullptr, nullptr};
        try {
            lane_bind_thread(c);
            int lane = 0;                                   // next lane to fill; when both are busy it holds the older slab
            std::vector<RowSeg> sg(job.lib_ids.size());
            auto finish = [&](int l) {
                const double t_in = now_s(); lane_wait(c, l); g_ns_gpu_wait += (uint64_t)((now_s() - t_in) * 1e9);
                Slab *S = fly[l]; fly[l] = nullptr;
                if (counts) {                               // the segments this slab appended to the row stores
                    lane_rows_segments(c, l, sg.data());
                    std::lock_guard<std::mutex> g(seg_m);
                    for (size_t li = 0; li < sg.size(); li++) { sg[li].seq = S->seq; sg[li].ctx = ctx_index; segs[li].push_back(sg[li]); }
                    if (!per_read) S->called = sg[0].called;
                }
                if (tenx) lane_cb_counters(c, l, S->cbn);
                after_gpu(S);
            };
            for (;;) {
                Slab *S = nullptr;
                if (fly[0] || fly[1]) {
                    if (!to_gpu.try_pop(S)) { finish(fly[lane] ? lane : lane ^ 1); continue; }   // nothing queued: retire the oldest
                } else if (!to_gpu.pop(S)) break;
                if (ab.flag) { to_commit.push(S); continue; }
                if (fly[lane]) finish(lane);
                fly[lane] = S;
                const double t_in = now_s();
                lane_submit(c, lane, &S->r1, S->paired ? &S->r2 : nullptr, job.lib_ids.data(), (int)job.lib_ids.size(),
                            S->res.empty() ? nullptr : S->res.data(), S->feats.empty() ? nullptr : S->feats.data(),
                            S->lt1.empty() ? nullptr : S->lt1.data(), (S->paired && !S->lt2.empty()) ? S->lt2.data() : nullptr,
                            counts ? S->key : nullptr, tenx ? S->cbc : nullptr, tenx ? S->cbq : nullptr, S->seq);
                g_ns_gpu_submit += (uint64_t)((now_s() - t_in) * 1e9);
                lane ^= 1;
            }
        } catch (const std::exception &e) { ab.set(e.what()); }
        // after a failure: every slab still has to find its way back to the pool
        for (Slab *&S : fly) if (S) { to_commit.push(S); S = nullptr; }
        if (ab.flag) { Slab *S; while (to_gpu.pop(S)) to_commit.push(S); }
    }

    void commit_main() {
        try {
            std::map<uint64_t, Slab *> pending;
            uint64_t next = 0;
            uint64_t fnv = 1469598103934665603ull;
            auto mix = [&](const char *p, size_t n) {
                for (size_t i = 0; i < n; i++) { fnv ^= (unsigned char)p[i]; fnv *= 1099511628211ull; }
                fnv ^= 0xFF; fnv *= 1099511628211ull;
            };
            std::string bases;
            auto unpack = [&](const nb200_reads &r, size_t i) {
                const uint8_t *rec = r.packed + i * (size_t)r.stride;
                const uint64_t *seq = (const uint64_t *)rec;
                const uint32_t *nm = (const uint32_t *)(rec + (size_t)r.words * 8);
                bases.resize(r.len[i]);
                for (uint32_t j = 0; j < r.len[i]; j++)
                    bases[j] = ((nm[j >> 5] >> (j & 31)) & 1) ? 'N' : "ACGT"[(seq[j >> 5] >> (2 * (j & 31))) & 3];
            };
            Slab *S = nullptr;
            while (to_commit.pop(S)) {
                pending[S->seq] = S;
                while (!pending.empty() && pending.begin()->first == next) {
                    Slab *T = pending.begin()->second;
                    pending.erase(pending.begin());
                    next++;
                    if (!ab.flag) {
                        for (size_t li = 0; li < libs.size(); li++) {
                            LibOut &lo = libs[li];
                            if (T->has_tags) {
                                const double t_in = now_s();
                                struct Acc { double t; ~Acc() { g_ns_write += (uint64_t)((now_s() - t) * 1e9); } } acc{t_in};
                                if (lo.f && !T->out[li].empty() && fwrite(T->out[li].data(), 1, T->out[li].size(), lo.f) != T->out[li].size()) throw IoError("write failed: " + lo.tmp);
                            } else {
                                for (auto &kv : T->bulk[li]) lo.bulk[kv.first] += kv.second;
                            }
                            std::string().swap(T->out[li]);
                        }
                        stats.n_reads += T->n; stats.bases1 += T->bases1; stats.bases2 += T->bases2; stats.called += T->called;
                        stats.paired |= T->paired; stats.has_tags |= T->has_tags; stats.n_slabs++;
                        tagged += T->tagged;
                        if (tenx) {
                            nb200_cb_stats &c = stats.cb;
                            c.total_pairs += T->pairs; c.name_mismatch += T->name_mismatch; c.too_short += T->too_short;
                            c.no_remaining_seq += T->no_remaining_seq;
                            c.cb_perfect_match += T->cbn[0]; c.cb_corrected += T->cbn[1]; c.cb_no_correction += T->cbn[2];
                            c.n_exact_miss += T->cbn[3]; c.n_multi += T->cbn[4]; c.probes += T->cbn[5];
                            c.written_pairs += T->cbn[0] + T->cbn[1];
                        }
                        if (dry && !getenv("NB200_INGEST_NOSUM"))      // reader statistics (nb200_host_ingest_stats): FNV-1a over every field of every read
                            for (size_t i = 0; i < T->n; i++) {
                                mix(T->names.ptr(i), T->names.len(i));
                                unpack(T->r1, i); mix(bases.data(), bases.size());
                                if (T->paired) { unpack(T->r2, i); mix(bases.data(), bases.size()); }
                                if (T->has_tags) { mix(T->cb.ptr(i), T->cb.len(i)); mix(T->ub.ptr(i), T->ub.len(i)); }
                            }
                    }
                    T->called = 0;
                    free_slabs.push(T);
                }
            }
            stats.checksum = fnv;
        } catch (const IoError &e) { ab.set(e.what(), true); drain(); } catch (const std::exception &e) { ab.set(e.what()); drain(); }
    }
    void drain() { Slab *S; while (to_commit.pop(S)) free_slabs.push(S); }

    // walker side: a full task gets a slab and goes to the pool
    uint64_t issued = 0;
    void dispatch(std::shared_ptr<Task> t) {
        if (t->e.empty() && t->segs.empty()) return;
        Slab *S = nullptr;
        const double t0 = now_s();
        if (!free_slabs.pop(S)) throw std::runtime_error("slab pool closed");
        g_wait_slab += now_s() - t0;
        if (ab.flag) { free_slabs.push(S); throw std::runtime_error(ab.what); }
        if (t->paired) need_mate2(S);
        S->seq = issued++;
        t->slab = S;
        t->trims = trims.empty() ? nullptr : &trims;
        t->bc = counts ? &bc : nullptr;
        if (tenx) { t->cb_len = job.cb_len; t->umi_len = job.umi_len; }
        pool->push(Pool::PARSE, [this, t] {
            const double t_in = now_s();
            try { parse_task(*t); } catch (...) { to_commit.push(t->slab); throw; }
            g_ns_parse += (uint64_t)((now_s() - t_in) * 1e9);
            after_parse(t->slab);
        });
    }
};

static size_t slab_room(uint32_t max_len) { return std::min(kSlabReads, kSlabSeqBytes / stride_for(max_len)); }

static void walk_bam(Pipeline &P, ByteSource &src) {
    Cursor cur(&src);
    auto task = std::make_shared<Task>();
    task->bam = true;
    cur.attach(&task->keep);
    {
        auto must = [&](size_t n) -> const unsigned char * {
            const char *p = cur.need(n, "BAM header");
            if (!p) throw IoError("truncated BAM header in " + P.job.inputs[0]);
            return (const unsigned char *)p;
        };
        const char *h = cur.need(4, "BAM header");
        if (!h || memcmp(h, "BAM\1", 4) != 0) throw std::runtime_error(P.job.inputs[0] + " is not a BAM file");
        size_t l_text = le32(must(4));
        while (l_text) { const size_t step = std::min<size_t>(l_text, 1u << 20); must(step); l_text -= step; }
        const uint32_t n_ref = le32(must(4));
        for (uint32_t i = 0; i < n_ref; i++) { const uint32_t l_name = le32(must(4)); must((size_t)l_name + 4); }
    }
    task->keep.blocks.clear(); task->keep.side.clear();
    cur.attach(&task->keep);
    bool first = true, file_paired = false;
    struct Open { std::shared_ptr<std::string> rec; uint64_t order; int which; };
    std::unordered_multimap<uint64_t, Open> open;         // mates waiting for their partner, by name hash
    const char *pend = nullptr; uint32_t pend_size = 0; int pend_which = 0;   // the previous record, when it waits for its mate
    uint64_t order = 0;
    auto name_of = [](const char *body, const unsigned char *&nm, uint32_t &len) { nm = (const unsigned char *)body + 32; const uint32_t l = (unsigned char)body[8]; len = l ? l - 1 : 0; };
    auto hash_name = [](const unsigned char *p, uint32_t n) { uint64_t x = 1469598103934665603ull; for (uint32_t j = 0; j < n; j++) { x ^= p[j]; x *= 1099511628211ull; } return x; };
    // entries being assembled may point into the last blocks / boundary copies of the task that is dispatched
    auto inherit = [](const Keep &from, Keep &to) {
        for (size_t i = from.blocks.size() > 2 ? from.blocks.size() - 2 : 0; i < from.blocks.size(); i++) to.blocks.push_back(from.blocks[i]);
        for (size_t i = from.side.size() > 4 ? from.side.size() - 4 : 0; i < from.side.size(); i++) to.side.push_back(from.side[i]);
    };
    auto flush = [&]() {
        auto nt = std::make_shared<Task>();
        nt->bam = true; nt->paired = file_paired;
        inherit(task->keep, nt->keep);
        P.dispatch(task);
        task = nt;
        cur.attach(&task->keep);
    };
    size_t room = slab_room(1);
    task->e.reserve(kSlabReads);
    auto emit = [&](const char *a, uint32_t la, const char *b, uint32_t lb) {
        const uint32_t L1 = a ? le32((const unsigned char *)a + 16) : 0, L2 = b ? le32((const unsigned char *)b + 16) : 0;
        if (L1 > task->max1 || L2 > task->max2) {
            if (L1 > NB200_MAX_READ_LEN || L2 > NB200_MAX_READ_LEN) throw std::runtime_error("read longer than 500 bases");
            room = slab_room(std::max(std::max(task->max1, L1), std::max(task->max2, L2)));
        }
        if (task->e.size() + 1 > room) {
            flush();
            task->e.reserve(kSlabReads);
            room = slab_room(std::max(L1, L2));
        }
        task->max1 = std::max(task->max1, L1); task->max2 = std::max(task->max2, L2);
        Entry e; e.a = a; e.la = la; e.b = b; e.lb = lb;
        task->e.push_back(e);
    };
    auto to_open = [&](const char *body, uint32_t size, int which) {
        const unsigned char *nm; uint32_t nl;
        name_of(body, nm, nl);
        open.emplace(hash_name(nm, nl), Open{std::make_shared<std::string>(body, size), order++, which});
    };
    for (;;) {
        const char *bs = cur.need(4, "BAM record");
        if (!bs) break;
        const uint32_t size = le32((const unsigned char *)bs);
        if (size < 32) throw std::runtime_error("truncated BAM record in " + P.job.inputs[0]);
        const char *body = cur.need(size, "BAM record");
        if (!body) throw IoError("truncated BAM record in " + P.job.inputs[0]);
        // the walk is a pointer chase through memory another core just wrote: fetch ahead where the next records
        // will be if they are about as long as this one
        __builtin_prefetch(body + 4 * (size_t)(size + 4));
        __builtin_prefetch(body + 4 * (size_t)(size + 4) + 64);
        __builtin_prefetch(body + 8 * (size_t)(size + 4));
        __builtin_prefetch(body + 8 * (size_t)(size + 4) + 64);
        const uint32_t flag = (unsigned char)body[14] | ((unsigned char)body[15] << 8);
        if (flag & 0x900) continue;                       // secondary / supplementary
        if (first) { first = false; file_paired = (flag & 1) != 0; task->paired = file_paired; }
        const int which = (flag & 0x80) ? 1 : 0;
        if (!file_paired) {
            // single-end file: every primary record is a read.  The walk stays minimal (size chain, flag, length); records
            // that lie back to back in a block form one run, a record straddling two blocks is a run of its own (`need`
            // made a contiguous copy of its body; its size field is copied in front of it)
            auto add_record = [&](const char *hdr, const char *bd, uint32_t sz) {
                const uint32_t L1 = le32((const unsigned char *)bd + 16);
                if (L1 > NB200_MAX_READ_LEN) throw std::runtime_error("read longer than 500 bases");
                if (L1 > task->max1) room = slab_room(L1);
                if (task->n_seg_records + 1 > room) { flush(); room = slab_room(L1); }
                task->max1 = std::max(task->max1, L1);
                if (bd != hdr + 4) {                 // header and body not contiguous: one joined copy
                    auto joined = std::make_shared<std::string>();
                    joined->reserve(4 + (size_t)sz);
                    joined->append(hdr, 4); joined->append(bd, sz);
                    task->keep.side.push_back(joined);
                    task->segs.push_back(Task::Seg{joined->data(), 1});
                } else if (!task->segs.empty() && task->segs.back().p + task->seg_bytes_of_last == hdr) {
                    task->segs.back().n++;
                    task->seg_bytes_of_last += 4 + (size_t)sz;
                    task->n_seg_records++;
                    return;
                } else {
                    task->segs.push_back(Task::Seg{hdr, 1});
                }
                task->seg_bytes_of_last = (bd != hdr + 4) ? 0 : 4 + (size_t)sz;      // (a joined copy is never extended)
                task->n_seg_records++;
            };
            add_record(bs, body, size);
            for (;;) {
                const char *h2 = cur.need(4, "BAM record");
                if (!h2) break;
                const uint32_t sz = le32((const unsigned char *)h2);
                if (sz < 32) throw std::runtime_error("truncated BAM record in " + P.job.inputs[0]);
                const char *b2 = cur.need(sz, "BAM record");
                if (!b2) throw IoError("truncated BAM record in " + P.job.inputs[0]);
                // the chain is a pointer chase through memory another core just wrote; records of 10x data are nearly all the
                // same size, so the headers 12 / 24 records ahead are about here
                __builtin_prefetch(b2 + 12 * (size_t)(sz + 4));
                __builtin_prefetch(b2 + 12 * (size_t)(sz + 4) + 64);
                __builtin_prefetch(b2 + 24 * (size_t)(sz + 4));
                __builtin_prefetch(b2 + 24 * (size_t)(sz + 4) + 64);
                const uint32_t fl = (unsigned char)b2[14] | ((unsigned char)b2[15] << 8);
                if (fl & 0x900) continue;                    // secondary / supplementary: ends the run (the next record starts a new one)
                add_record(h2, b2, sz);
            }
            P.dispatch(task);
            return;
        }
        if (!(flag & 1)) {                                // unpaired record inside a paired file: a singleton
            if (which) emit(nullptr, 0, body, size); else emit(body, size, nullptr, 0);
            continue;
        }
        const unsigned char *nm; uint32_t nl;
        name_of(body, nm, nl);
        if (pend) {
            const unsigned char *pn; uint32_t pl;
            name_of(pend, pn, pl);
            if (pend_which != which && pl == nl && memcmp(pn, nm, nl) == 0) {
                if (which) emit(pend, pend_size, body, size); else emit(body, size, pend, pend_size);
                pend = nullptr;
                continue;
            }
            to_open(pend, pend_size, pend_which);
            pend = nullptr;
        }
        // its mate may have gone by earlier (coordinate-ordered input)
        bool matched = false;
        if (!open.empty()) {
            auto range = open.equal_range(hash_name(nm, nl));
            for (auto it = range.first; it != range.second; ++it) {
                const std::string &o = *it->second.rec;
                const unsigned char *on; uint32_t ol;
                name_of(o.data(), on, ol);
                if (it->second.which == which || ol != nl || memcmp(on, nm, nl) != 0) continue;
                task->keep.side.push_back(it->second.rec);        // (a flush inside emit hands the last copies on to the new task)
                if (which) emit(o.data(), (uint32_t)o.size(), body, size); else emit(body, size, o.data(), (uint32_t)o.size());
                open.erase(it);
                matched = true;
                break;
            }
        }
        if (!matched) { pend = body; pend_size = size; pend_which = which; }
    }
    if (pend) to_open(pend, pend_size, pend_which);
    // records whose mate never came: singletons, in the order they were read
    std::vector<Open> rest;
    for (auto &kv : open) rest.push_back(kv.second);
    std::sort(rest.begin(), rest.end(), [](const Open &x, const Open &y) { return x.order < y.order; });
    for (const Open &o : rest) {
        task->keep.side.push_back(o.rec);
        if (o.which) emit(nullptr, 0, o.rec->data(), (uint32_t)o.rec->size()); else emit(o.rec->data(), (uint32_t)o.rec->size(), nullptr, 0);
    }
    P.dispatch(task);
}

static void walk_fastq(Pipeline &P, ByteSource &s1, ByteSource *s2) {
    Cursor c1(&s1);
    std::unique_ptr<Cursor> c2(s2 ? new Cursor(s2) : nullptr);
    auto task = std::make_shared<Task>();
    task->paired = s2 != nullptr;
    auto attach = [&] { c1.attach(&task->keep); if (c2) c2->attach(&task->keep); };
    attach();
    const bool want_q = !P.trims.empty() || P.tenx;
    // 10x mode reads FASTQ as fastq-to-bam does (load_fastq_qual): blank lines between records, a '+' line, qualities as
    // long as the sequence; read lengths are checked after the barcode and UMI are cut off (tenx_select)
    const bool tenx = P.tenx;
    auto record = [&](Cursor &c, const std::string &path, const char *&name, uint32_t &nl, const char *&seq, uint32_t &sl, const char *&qual) -> bool {
        qual = nullptr;
        const char *p; size_t n;
        if (!c.line(p, n)) return false;
        if (n == 0 && !c.line(p, n)) return false;          // tolerate one blank line at the end
        while (tenx && n == 0) if (!c.line(p, n)) return false;
        if (n == 0 || p[0] != '@') throw std::runtime_error("malformed FASTQ record in " + path);
        size_t e = 1;
        while (e < n && p[e] != ' ' && p[e] != '\t') e++;
        name = p + 1; nl = (uint32_t)(e - 1);
        if (!c.line(p, n)) throw std::runtime_error("truncated FASTQ record in " + path);
        if (n > NB200_MAX_READ_LEN && !tenx) throw std::runtime_error("read longer than 500 bases");
        seq = p; sl = (uint32_t)n;
        const char *q; size_t qn;
        if (tenx) {
            if (!c.line(q, qn)) throw std::runtime_error("truncated FASTQ record in " + path);
            if (qn == 0 || q[0] != '+') throw std::runtime_error("malformed FASTQ record (no '+' line) in " + path);
            if (!c.line(q, qn)) { q = p; qn = 0; }          // empty quality line at the end of the file
            if (qn != sl) throw std::runtime_error("FASTQ sequence and quality lengths differ in " + path);
            qual = q;
            return true;
        }
        if (!c.line(q, qn)) return true;                    // '+' line and qualities may be missing at the very end
        if (c.line(q, qn) && want_q && qn == sl) qual = q;  // (a quality line of another length is ignored: no trimming)
        return true;
    };
    // 10x mode: the longest read the slab will hold of this pair (over-long reads fail in the parse task)
    const uint32_t bl = tenx ? (uint32_t)(P.job.cb_len + P.job.umi_len) : 0;
    auto held = [&](uint32_t len, uint32_t cut) { return tenx ? std::min<uint32_t>(len > cut ? len - cut : 0, NB200_MAX_READ_LEN) : len; };
    for (;;) {
        Entry e;
        const char *nm; uint32_t nl;
        if (!record(c1, P.job.inputs[0], nm, nl, e.a, e.la, e.qa)) break;
        e.name = nm; e.ln = nl;
        if (c2) {
            const char *n2; uint32_t l2;
            if (!record(*c2, P.job.inputs[1], n2, l2, e.b, e.lb, e.qb)) {
                if (!tenx) throw std::runtime_error("R1 and R2 FASTQ files hold different numbers of reads");
                // fastq-to-bam zips the two files: pairs stop at the shorter one, the rest of R1 is only checked
                Keep rest;
                c1.attach(&rest);
                while (record(c1, P.job.inputs[0], nm, nl, e.a, e.la, e.qa)) { rest.blocks.clear(); rest.side.clear(); }
                c2.reset();
                break;
            }
            e.name2 = n2; e.ln2 = l2;
        }
        const uint32_t m1 = std::max(task->max1, held(e.la, bl)), m2 = std::max(task->max2, held(e.lb, 0));
        if (task->e.size() + 1 > slab_room(std::max(m1, m2))) {
            auto nt = std::make_shared<Task>();
            nt->paired = task->paired;
            // e points into blocks / boundary copies registered with the old task: the new one keeps the last of them alive
            for (size_t i = task->keep.blocks.size() > 4 ? task->keep.blocks.size() - 4 : 0; i < task->keep.blocks.size(); i++) nt->keep.blocks.push_back(task->keep.blocks[i]);
            for (size_t i = task->keep.side.size() > 8 ? task->keep.side.size() - 8 : 0; i < task->keep.side.size(); i++) nt->keep.side.push_back(task->keep.side[i]);
            P.dispatch(task);
            task = nt;
            attach();
        }
        task->max1 = std::max(task->max1, held(e.la, bl)); task->max2 = std::max(task->max2, held(e.lb, 0));
        task->e.push_back(e);
    }
    if (c2) {
        const char *n2; uint32_t l2; const char *sq; uint32_t sl; const char *qq;
        Keep rest;
        if (tenx) c2->attach(&rest);
        while (record(*c2, P.job.inputs[1], n2, l2, sq, sl, qq)) {
            if (!tenx) throw std::runtime_error("R1 and R2 FASTQ files hold different numbers of reads");
            rest.blocks.clear(); rest.side.clear();        // 10x mode: the rest of R2 is only checked (zip)
        }
    }
    P.dispatch(task);
}

}  // namespace

}  // namespace nb200

// test hook (host only): the raw-DEFLATE decoder of the BGZF reader; 1 = decoded into exactly out_len bytes
extern "C" int32_t nb200_fast_inflate(const uint8_t *in, uint64_t in_len, uint8_t *out, uint64_t out_len) {
    return nb200::fast_inflate(in, (size_t)in_len, out, (size_t)out_len) ? 1 : 0;
}

namespace nb200 {

void run_file_pipeline(const FileJob &job, FileStats *stats_out) {
    if (job.inputs.empty() || job.inputs.size() > 2) throw std::runtime_error("expected one or two --input files");
    const bool counts = !job.counts_outputs.empty();
    if (!job.ctxs.empty() && (job.lib_ids.empty() || (!job.outputs.empty() && job.lib_ids.size() != job.outputs.size()) ||
                              (job.outputs.empty() && !counts) || (counts && job.counts_outputs.size() != job.lib_ids.size())))
        throw std::runtime_error("bad arguments");
    const auto t0 = std::chrono::steady_clock::now();
    Pipeline P(job);
    P.dry = job.ctxs.empty();
    P.counts = counts && !P.dry;
    P.per_read = !job.outputs.empty();
    P.tenx = job.whitelist != nullptr;
    if (P.tenx && (!P.counts || P.per_read || job.inputs.size() != 2 || job.umi_len < 0))
        throw std::runtime_error("bad arguments");
    g_wait_block = g_wait_slab = 0.0;
    g_ns_inflate = 0; g_ns_parse = 0; g_ns_format = 0; g_ns_gpu_wait = 0; g_ns_gpu_submit = 0; g_ns_write = 0; g_ns_intern = 0;
    double t_alloc = 0.0, t_walk = 0.0, t_drain = 0.0, t_finish = 0.0, t_free = 0.0, t_counts = 0.0;
    const int T = std::max(1, job.host_threads);
    const bool bam = ends_with_ci(job.inputs[0], ".bam");
    if (bam && job.inputs.size() != 1) throw std::runtime_error("one BAM file expected");
    if (P.counts && !bam && !P.tenx)
        throw std::runtime_error("counts need cell barcodes and UMIs (CB / UB tags of a BAM file); " + job.inputs[0] + " is FASTQ: write the per-read TSV instead");
    if (P.tenx && bam) throw std::runtime_error("fastq-to-counts reads raw R1 / R2 FASTQ files; " + job.inputs[0] + " is a BAM file");
    if (P.counts) {                                    // (feature names the per-read TSV cannot carry fail here, before any work)
        for (nb200_ctx *c : job.ctxs) lane_rows_begin(c, job.lib_ids.data(), (int)job.lib_ids.size());
        P.segs.resize(job.lib_ids.size());
    }
    std::vector<uint32_t> wl_rank;                     // 10x mode: whitelist line -> cell rank (lane_cb_begin)
    std::vector<std::string> wl_cells;
    struct CbEnd { const FileJob &j; bool on; ~CbEnd() { if (on) try { lane_cb_end(j.ctxs); } catch (...) {} } } cb_end{job, P.tenx};
    if (P.tenx) lane_cb_begin(job.ctxs, *job.whitelist, job.cb_len, &wl_rank, &wl_cells);
    // outputs
    for (size_t li = 0; li < (P.dry ? 0 : job.lib_ids.size()); li++) {
        LibOut lo;
        lo.lib_id = job.lib_ids[li];
        lo.max_hits = lane_max_hits(job.ctxs[0], lo.lib_id);
        if (P.per_read) { lo.path = job.outputs[li]; lo.tmp = lo.path + ".tmp"; }
        lo.gz = ends_with_ci(lo.path, ".gz");
        const uint32_t nf = lane_n_features(job.ctxs[0], lo.lib_id);
        lo.names.resize(nf);
        for (uint32_t f = 0; f < nf; f++) { uint32_t len; const char *p = lane_feature_name(job.ctxs[0], lo.lib_id, f, &len); lo.names[f] = {p, len}; }
        P.libs.push_back(std::move(lo));
    }
    if (!P.dry) {
        bool any = false;
        for (int32_t id : job.lib_ids) { int t; double st; any |= lane_trim(job.ctxs[0], id, &t, &st); }
        if (any) {
            P.trims.resize(job.lib_ids.size());
            for (size_t li = 0; li < job.lib_ids.size(); li++) { int t; double st; if (lane_trim(job.ctxs[0], job.lib_ids[li], &t, &st)) P.trims[li].init(t, st); }
        }
    }
    try {
        if (!P.dry) lane_bind_thread(job.ctxs[0]);
        P.pool.reset(new Pool(T, P.ab));
        const size_t n_slabs = (P.dry ? 2 : 3 * job.ctxs.size()) + (size_t)std::min(T, 64) + 2;
        { const double ta = now_s(); P.start_pool(n_slabs, P.dry ? nullptr : job.ctxs[0]); t_alloc = now_s() - ta; }
        for (LibOut &lo : P.libs) {
            if (!P.per_read) break;
            lo.f = fopen(lo.tmp.c_str(), "wb");
            if (!lo.f) throw IoError("cannot write " + lo.tmp);
            if (bam) {                                      // per-read TSV: the header leads (its own gzip member for .gz)
                std::string hdr(kPerReadHeader), z;
                if (lo.gz) gzip_member(hdr, z);
                const std::string &w = lo.gz ? z : hdr;
                if (fwrite(w.data(), 1, w.size(), lo.f) != w.size()) throw IoError("write failed: " + lo.tmp);
            }
        }
        for (size_t d = 0; d < job.ctxs.size(); d++) P.gpu_threads.emplace_back([&P, &job, d] { P.gpu_main(job.ctxs[d], (int)d); });
        P.committer = std::thread([&P] { P.commit_main(); });
        std::string walk_err; bool walk_io = false;
        const double tw = now_s();
        try {
            if (bam) {
                std::unique_ptr<ByteSource> src;
                if (BgzfSource::is_bgzf(job.inputs[0])) src.reset(new BgzfSource(job.inputs[0], *P.pool, P.ab, T + 4));      // chunks inflated ahead of the walker: parse / format tasks go first in the pool, so a short window starves it
                else src.reset(new GzSource(job.inputs[0], P.ab));           // one gzip member (e.g. python's gzip module)
                walk_bam(P, *src);
            } else {
                auto open_src = [&](const std::string &p) -> std::unique_ptr<ByteSource> {
                    if (ends_with_ci(p, ".gz") && BgzfSource::is_bgzf(p)) return std::unique_ptr<ByteSource>(new BgzfSource(p, *P.pool, P.ab, T / 4 + 2));
                    return std::unique_ptr<ByteSource>(new GzSource(p, P.ab));
                };
                std::unique_ptr<ByteSource> a = open_src(job.inputs[0]), b;
                if (job.inputs.size() == 2) b = open_src(job.inputs[1]);
                walk_fastq(P, *a, b.get());
            }
        } catch (const IoError &e) { walk_err = e.what(); walk_io = true; } catch (const std::exception &e) { walk_err = e.what(); }
        t_walk = now_s() - tw;
        if (!walk_err.empty()) P.ab.set(walk_err, walk_io);
        P.stop_pinner();
        const double t_drain0 = now_s();
        // wait until every issued slab has come back through the committer
        {
            std::vector<Slab *> got;
            while (got.size() < P.slabs.size()) { Slab *S; if (!P.free_slabs.pop(S)) break; got.push_back(S); }
        }
        P.to_gpu.close();
        for (auto &t : P.gpu_threads) t.join();
        P.gpu_threads.clear();
        P.to_commit.close();
        P.committer.join();
        P.pool->stop();
        t_drain = now_s() - t_drain0;
        const double t_fin0 = now_s();
        if (P.ab.flag) {
            for (LibOut &lo : P.libs) { if (lo.f) fclose(lo.f); lo.f = nullptr; remove(lo.tmp.c_str()); }
            P.free_all();
            if (P.ab.io) throw IoError(P.ab.what);
            throw std::runtime_error(P.ab.what);
        }
        if (P.counts && !P.tenx && P.stats.n_reads && !P.tagged)
            throw std::runtime_error("no read of " + job.inputs[0] + " carries a CB or UB tag: counts need cell barcodes and UMIs");
        // finish the files: per-read outputs are complete, bulk tables are written now
        for (LibOut &lo : P.libs) {
            if (!lo.f) continue;
            if (!bam) {
                // `features<TAB>count` for untagged input (nimble/parse.py:39-57), rows in ascending feature-string order
                std::vector<std::pair<std::string, uint64_t>> rows;
                rows.reserve(lo.bulk.size());
                for (auto &kv : lo.bulk) {
                    std::string nm;
                    const int32_t *ids = (const int32_t *)kv.first.data();
                    for (size_t j = 0; j < kv.first.size() / 4; j++) { if (j) nm += ','; nm.append(lo.names[(size_t)ids[j]].first, lo.names[(size_t)ids[j]].second); }
                    rows.emplace_back(std::move(nm), kv.second);
                }
                std::sort(rows.begin(), rows.end());
                std::string text = "nimble_features\tnimble_score\n";
                for (auto &r : rows) { text += r.first; text += '\t'; put_uint(text, r.second); text += '\n'; }
                std::string z;
                if (lo.gz) gzip_member(text, z);
                const std::string &w = lo.gz ? z : text;
                if (fwrite(w.data(), 1, w.size(), lo.f) != w.size()) throw IoError("write failed: " + lo.tmp);
            }
            if (fclose(lo.f) != 0) { lo.f = nullptr; throw IoError("write failed: " + lo.tmp); }
            lo.f = nullptr;
            if (rename(lo.tmp.c_str(), lo.path.c_str()) != 0) throw IoError("cannot rename " + lo.tmp);
        }
        t_finish = now_s() - t_fin0;
        if (P.counts) {
            // counts TSVs (nimble/__main__.py:254-293): every library's rows gathered in slab order on the first context,
            // cells ranked by CB bytes, the UMI stage on the device
            const double tc = now_s();
            std::vector<uint32_t> rank;
            std::vector<std::string> cells;
            if (P.tenx) {                                   // cells are whitelist lines; the cache rule decides the open ones
                lane_cb_resolve(job.ctxs);
                rank.swap(wl_rank); cells.swap(wl_cells);
            } else {
                std::vector<std::string> cell_names = P.bc.cell_names();
                std::vector<uint32_t> order(cell_names.size());
                rank.resize(cell_names.size()); cells.resize(cell_names.size());
                for (uint32_t i = 0; i < order.size(); i++) order[i] = i;
                std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return cell_names[a] < cell_names[b]; });
                for (uint32_t r = 0; r < order.size(); r++) { rank[order[r]] = r; cells[r] = std::move(cell_names[order[r]]); }
            }
            for (size_t li = 0; li < P.libs.size(); li++) {
                std::vector<RowSeg> &sg = P.segs[li];
                std::sort(sg.begin(), sg.end(), [](const RowSeg &a, const RowSeg &b) { return a.seq < b.seq; });
                nb200_counts table{};
                uint64_t rows = 0;
                lane_rows_count(job.ctxs, (int)li, job.lib_ids[li], sg, rank, job.umi_threshold, job.umi_flags, &table, &rows, P.tenx);
                std::vector<std::string> names(P.libs[li].names.size());
                for (size_t f = 0; f < names.size(); f++) names[f].assign(P.libs[li].names[f].first, P.libs[li].names[f].second);
                write_counts_tsv(job.counts_outputs[li], table.n_rows ? &table : nullptr, names, cells);
                P.stats.counts3.push_back(rows); P.stats.counts3.push_back(table.n_rows); P.stats.counts3.push_back(table.dropped_empty);
                if (job.umi_flags & NB200_UMI_CORRECT) {
                    uint64_t corrected = 0;
                    nb200_umis_corrected(job.ctxs[0], &corrected);
                    P.stats.counts3.push_back(corrected);
                }
            }
            lane_bind_thread(job.ctxs[0]);
            t_counts = now_s() - tc;
        }
        const double t_free0 = now_s();
        P.free_all();
        t_free = now_s() - t_free0;
    } catch (...) {
        P.ab.set("aborted");
        P.stop_pinner();
        P.free_slabs.close(); P.to_gpu.close();
        for (auto &t : P.gpu_threads) if (t.joinable()) t.join();
        P.to_commit.close();
        if (P.committer.joinable()) P.committer.join();
        if (P.pool) P.pool->stop();
        for (LibOut &lo : P.libs) if (lo.f) { fclose(lo.f); remove(lo.tmp.c_str()); }
        P.free_all();
        throw;
    }
    P.stats.seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    if (getenv("NB200_TRACE"))
        fprintf(stderr, "[nb200 trace] pipeline: %.3f s total | slab pool %.3f | walker %.3f (waiting for blocks %.3f, for slabs %.3f) | drain %.3f | close+rename %.3f | free slabs %.3f | %llu slabs | "
                        "pool thread-seconds: inflate %.3f parse %.3f (barcode keys %.3f) format %.3f | gpu threads: submit %.3f wait %.3f | writer %.3f | counts %.3f\n",
                P.stats.seconds, t_alloc, t_walk, g_wait_block, g_wait_slab, t_drain, t_finish, t_free, (unsigned long long)P.stats.n_slabs,
                g_ns_inflate.load() * 1e-9, g_ns_parse.load() * 1e-9, g_ns_intern.load() * 1e-9, g_ns_format.load() * 1e-9, g_ns_gpu_submit.load() * 1e-9,
                g_ns_gpu_wait.load() * 1e-9, g_ns_write.load() * 1e-9, t_counts);
    if (stats_out) *stats_out = P.stats;
}

}  // namespace nb200
