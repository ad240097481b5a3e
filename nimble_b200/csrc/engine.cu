// nimble_b200 engine: context, HBM residency, streamed ingest, pipelined kernel batches, C ABI.
// Reference boundary replaced: nimble/__main__.py:153-211 (align -> exec aligner) and
// nimble/__main__.py:254-293 (report).  See include/nimble_b200.h for the per-entry citations.
#include <algorithm>
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <chrono>
#include <cstring>
#include <functional>
#include <memory>
#include <stdexcept>
#include <string>
#include <thread>
#include <type_traits>
#include <unordered_set>
#include <vector>

#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>
#include <cuda_runtime.h>

#include "../../include/nimble_b200.h"
#include "agg.cuh"
#include "barcode.cuh"
#include "checksum.hpp"
#include "kernels.cuh"
#include "ingest.hpp"
#include "library.hpp"
#include "pandas_na.hpp"
#include "slab_api.hpp"
#include "stream.hpp"
#include "trim.hpp"

namespace nb200 {

struct CudaError : std::runtime_error { using std::runtime_error::runtime_error; };

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            throw CudaError(std::string(#call) + ": " + cudaGetErrorString(e_));                   \
    } while (0)

// Device memory with one owner: freed by its destructor, handed on only by moving.  A buffer is freed with whatever device
// is current, so code that frees another device's buffers sets that device first.
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(DevBuf &&o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
    DevBuf &operator=(DevBuf &&o) noexcept {
        if (this != &o) { release(); p = o.p; cap = o.cap; o.p = nullptr; o.cap = 0; }
        return *this;
    }
    ~DevBuf() { release(); }
    void ensure(size_t bytes) {
        if (bytes <= cap) return;
        if (p) CK(cudaFree(p));
        p = nullptr; cap = 0;
        size_t want = bytes + bytes / 8 + 256;
        CK(cudaMalloc(&p, want));
        cap = want;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};
static_assert(!std::is_copy_constructible<DevBuf>::value && !std::is_copy_assignable<DevBuf>::value &&
                  std::is_nothrow_move_constructible<DevBuf>::value,
              "a DevBuf has one owner; std::vector<DevBuf> moves its elements");

// Pinned host memory for `cap` elements of T, owned like a DevBuf.  ensure() allocates exactly what it is asked for.
template <class T> struct PinnedBuf {
    T *p = nullptr;
    size_t cap = 0;
    PinnedBuf() = default;
    PinnedBuf(PinnedBuf &&o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
    PinnedBuf &operator=(PinnedBuf &&o) noexcept {
        if (this != &o) { release(); p = o.p; cap = o.cap; o.p = nullptr; o.cap = 0; }
        return *this;
    }
    ~PinnedBuf() { release(); }
    void ensure(size_t count) {
        if (count <= cap) return;
        release();
        CK(cudaMallocHost(&p, count * sizeof(T)));
        cap = count;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

// A CUDA stream or event with one owner; converts to the raw handle, so it is passed to the runtime as one.
template <class H, cudaError_t (*Destroy)(H)> struct CudaHandle {
    H h = nullptr;
    CudaHandle() = default;
    CudaHandle(CudaHandle &&o) noexcept : h(o.h) { o.h = nullptr; }
    CudaHandle &operator=(CudaHandle &&o) noexcept {
        if (this != &o) { if (h) Destroy(h); h = o.h; o.h = nullptr; }
        return *this;
    }
    ~CudaHandle() { if (h) Destroy(h); }
    operator H() const { return h; }
};
using Stream = CudaHandle<cudaStream_t, cudaStreamDestroy>;
using Event = CudaHandle<cudaEvent_t, cudaEventDestroy>;

struct DevLibrary {
    HostLibrary host;
    LibDev dev{};
    DevBuf slab;             // table | class bitsets | positions | refs: one range for the L2 persistence window
    DevBuf tok_end, tok_comma;
    DevBuf min_score;        // score_percent as a per-length table (call_params), rebuilt when score_percent changes
    double min_score_for = 0.0;
    bool min_score_ok = false;
    bool probe_warp = false;     // NB200_PROBE_WARP=1: every read through the warp-per-read probe (the in-tree reference)
    size_t table_bytes = 0, slab_bytes = 0;
};

struct DevWhitelist {
    std::vector<std::string> entries;      // every non-empty line, caller's order
    DevBuf table;
    WlDev dev{};
    uint64_t n_slots = 0, n_unique = 0;
    int cb_len = 16;
};

}  // namespace nb200

using namespace nb200;

struct nb200_ctx {
    int device = 0, host_threads = 1, sm_count = 148;
    size_t l2_persist_max = 0, l2_window_max = 0;
    const DevLibrary *l2_window_lib = nullptr;
    std::string err;
    Stream s_compute, s_copy[2];
    std::vector<Event> ev_pool;
    std::vector<std::unique_ptr<DevLibrary>> libs;
    // resident reads
    DevBuf d_r1, d_r1len, d_r2, d_r2len, d_key;
    DevBuf stage1, stage2, d_nidx, d_nmask;        // compact wire form: seq words as they arrive, side table of the reads with N
    ReadsDev r1{}, r2{};
    uint64_t n_reads = 0;
    bool paired = false, has_key = false, resident = false;
    // per batch
    // per-batch state, double-buffered: batch k's alignment/calling kernels (s_tail) overlap batch k+1's probe (s_compute)
    struct BatchBuf { DevBuf ro, roB, items, sw_pairs, sw_rep, deferred, wide_list, warp_list, sums, slow_list, setup_list; Counters *ctr = nullptr; Event tail_done, probe_done; bool busy = false; } bb[2];
    DevBuf wide_scratch, wide_v;
    // streaming file path: two slabs in flight, each with its own device buffers (slab_api.hpp)
    struct FileLane {
        DevBuf r1, l1, r2, l2;
        std::vector<DevBuf> res, feats, nf;       // per library of the call
        std::vector<DevBuf> l1v, l2v;             // per library: trimmed read lengths (--trim), else unused
        std::vector<uint16_t *> hlen1, hlen2;     // what was submitted (host pointers; empty = no trimming)
        Event h2d_done, done;
        PinnedBuf<Counters> h_ctr;                // one Counters per library (overflow of the SW work list)
        bool busy = false;
        nb200_reads hr1{}, hr2{};                 // what was submitted (an overflow re-runs it)
        bool paired = false;
        std::vector<int32_t> libs;
        std::vector<nb200_read_result *> out_res;
        std::vector<int32_t *> out_feats;
        // counts mode: the slab's keys, the segment record per library (device / pinned: row0, rows, id0, ids, called)
        DevBuf key, seg;
        PinnedBuf<unsigned long long> h_seg;
        const uint64_t *hkey = nullptr;           // what was submitted (an overflow re-runs it)
        uint64_t n_rows_max = 0;                  // reads of the slab in flight: bound on the rows it appends
        // fastq-to-counts: the slab's barcodes and their correction (cb_*: device; h_cb: pinned CbCounters + log end)
        DevBuf cb, cbq, cb_raw, cb_idx, cb_st, cb_miss, cb_multi, cb_ctr;
        const uint8_t *hcb = nullptr, *hcbq = nullptr;   // what was submitted (an overflow re-runs it)
        uint64_t seq = 0;
        PinnedBuf<unsigned long long> h_cb;
    } lane[kFileLanes];
    // fastq-to-counts (lane_cb_*): the whitelist table, and the log of reads with several candidates (raw barcode, file
    // order, own choice; tx_n = entries, device-side).  The log grows like the row stores: tx_hi = its end as of the
    // last slab the host has seen.  tx_dec (first context, lane_cb_resolve): the decision per entry of every log.
    DevBuf tx_table, tx_key, tx_ord, tx_choice, tx_n, tx_dec;
    WlDev tx_wl{};
    uint64_t tx_cap = 0, tx_hi = 0;
    std::vector<DevBuf> tx_old;
    std::vector<uint64_t> tx_base;                // first context: where each context's log starts in tx_dec
    // counts mode (slab_api.hpp): per library of the call, the rows that count, appended slab by slab on s_copy[1]
    struct RowStore {
        DevBuf key, nf, ids, hdr, na;             // hdr: rows / ids used (device); na: per feature, name is a pandas NA token
        uint64_t cap_rows = 0, cap_ids = 0;
        uint64_t hi_rows = 0, hi_ids = 0;         // store end as of the last segment the host has seen
        std::vector<DevBuf> old;                  // outgrown buffers: freed when the call is done with the store
        uint32_t mh = 1;
        void reset() {                            // empty, its rows and outgrown buffers freed (hdr and na stay)
            key.release(); nf.release(); ids.release();
            old.clear();
            cap_rows = cap_ids = hi_rows = hi_ids = 0;
        }
    };
    std::vector<RowStore> rs;
    DevBuf rs_val, rs_pos, rs_tmp, rs_rank;
    Stream s_tail;
    int overlap = 1, stats = 0, defer_fetch = 0;
    bool fetch_pending = false, fetch_started = false;   // a count table waits on the device for nb200_fetch_counts / its copies are in flight
    uint32_t items_cap = 0;
    // per read
    DevBuf results, feats, row_nf;
    int32_t feats_stride = 0;
    DevBuf d_ctr, d_ctr_odd;                      // Counters: bb[0].ctr is d_ctr, bb[1].ctr is d_ctr_odd
    // aggregation
    DevBuf flag, permA, permB, k32A, k32B, k64A, k64B, num, cub_tmp, gstart, head;
    DevBuf u_cell, u_n, u_list, s_rep, s_S, s_U, s_fs, s_fc, s_flags;
    DevBuf row_n, row_off, slow, htable, rep_of, is_rep, cell_ord, rank_of, gstart2;
    DevBuf umi_table, umi_key;                    // UMI correction (NB200_UMI_CORRECT): the slot table, the rewritten keys
    uint64_t umis_corrected = 0;                  // of the last UMI stage (nb200_umis_corrected)
    DevBuf o_cell_d, o_count_d, o_n_d, o_list_d, gen_feats, gen_nf, gen_off, gen_score, gen_key;
    // count table lives in pinned host memory owned by the context
    PinnedBuf<uint32_t> h_cell, h_count, h_off, h_ids;
    DevBuf o_off_d, o_ids_d;
    nb200_timing timing{};
    uint64_t launches = 0;
    uint64_t dev_rows = 0, dev_ids = 0;     // extent of the device-side count table (nb200_counts_device)
    // fastq-to-bam: whitelists + one resident barcode batch
    std::vector<std::unique_ptr<DevWhitelist>> wls;
    DevBuf cb_chars, cb_qual, cb_elig, cb_keys, cb_idx, cb_status, cb_inval, cb_inval_chars, cb_hit;
    DevBuf d_cbctr;                               // CbCounters
    uint64_t cb_n = 0;
    int cb_len = 0;
    bool cb_has_elig = false, cb_resident = false;
};

static thread_local std::string g_create_err;
constexpr int kWideBlocks = 64;   // persistent grid of the wide-read kernel (4 warps per block)

namespace nb200 {

static cudaEvent_t new_event(nb200_ctx *c) {
    Event e;
    CK(cudaEventCreate(&e.h));
    c->ev_pool.push_back(std::move(e));
    return c->ev_pool.back();
}

__global__ void end_batch_kernel(Counters *ctr) {
    const unsigned long long items = ctr->alloc & kItemMask;
    if (items > ctr->items_max) ctr->items_max = items;
    ctr->deferred_total += ctr->alloc >> 40;
    ctr->alloc = 0;
    ctr->wide_total += ctr->n_wide;
    ctr->n_wide = 0;
    ctr->probe_warp_total += ctr->n_probe_warp;
    ctr->n_probe_warp = 0;
    ctr->sw_items += items;
    ctr->n_swpairs = 0;
    ctr->n_slow = 0;
    ctr->n_setup = 0;
    ctr->n_warpdef = 0;
}

// odd batches count into their own Counters: fold them into the main one before the host reads it
__global__ void merge_counters_kernel(Counters *a, Counters *b) {
    const int t = threadIdx.x;
    if (t < kCtrSpread) { a->probes[t] += b->probes[t]; a->probe_slots[t] += b->probe_slots[t]; b->probes[t] = 0; b->probe_slots[t] = 0; }
    if (t == 0) {
        a->overflow += b->overflow; a->sw_pairs += b->sw_pairs; a->sw_cells += b->sw_cells; a->sw_dups += b->sw_dups;
        a->sw_items += b->sw_items; a->deferred_total += b->deferred_total; a->wide_total += b->wide_total;
        a->probe_warp_total += b->probe_warp_total; b->probe_warp_total = 0;
        if (b->max_nf > a->max_nf) a->max_nf = b->max_nf;
        if (b->items_max > a->items_max) a->items_max = b->items_max;
        b->overflow = 0; b->sw_pairs = 0; b->sw_cells = 0; b->sw_dups = 0; b->sw_items = 0; b->deferred_total = 0; b->wide_total = 0;
        b->max_nf = 0; b->items_max = 0;
    }
}

// Compact wire form (include/nimble_b200.h, nb200_reads): seq words only cross PCIe; the full record
// [seq u64 x words][nmask u32 x words][pad] is rebuilt here, N masks from the side table.
__global__ void expand_reads_kernel(uint64_t n, const uint64_t *__restrict__ src, uint32_t words, uint8_t *__restrict__ dst, uint32_t dstride) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t *s = src + i * words;
    uint64_t *d = reinterpret_cast<uint64_t *>(dst + i * dstride);
    const uint32_t total = dstride / 8;
    for (uint32_t t = 0; t < total; t++) d[t] = t < words ? s[t] : 0ull;
}
__global__ void scatter_nmask_kernel(uint32_t cnt, const uint32_t *__restrict__ idx, const uint32_t *__restrict__ mask, uint32_t words,
                                     uint8_t *__restrict__ dst, uint32_t dstride) {
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= cnt) return;
    uint32_t *nm = reinterpret_cast<uint32_t *>(dst + (uint64_t)idx[j] * dstride + (size_t)words * 8);
    for (uint32_t t = 0; t < words; t++) nm[t] = mask[(uint64_t)j * words + t];
}

static inline bool is_compact(const nb200_reads *r) { return r->stride == 8 * r->words; }
static inline uint32_t full_stride(uint32_t words) { return (12 * words + 15) & ~15u; }

// reads [r0, r0 + nb) of a host batch -> device records, in order on stream cs.  Returns the bytes sent.
static uint64_t h2d_reads(nb200_ctx *c, cudaStream_t cs, const nb200_reads *h, DevBuf &stage, uint8_t *d_rec, uint16_t *d_len,
                          uint64_t r0, uint64_t nb) {
    if (!nb) return 0;
    uint64_t bytes = nb * ((uint64_t)h->stride + 2);
    CK(cudaMemcpyAsync(d_len + r0, h->len + r0, nb * 2, cudaMemcpyHostToDevice, cs));
    if (!is_compact(h)) {
        CK(cudaMemcpyAsync(d_rec + r0 * h->stride, h->packed + r0 * h->stride, nb * (size_t)h->stride, cudaMemcpyHostToDevice, cs));
        return bytes;
    }
    const uint32_t ds = full_stride(h->words);
    stage.ensure(nb * (size_t)h->stride + 64);
    CK(cudaMemcpyAsync(stage.p, h->packed + r0 * h->stride, nb * (size_t)h->stride, cudaMemcpyHostToDevice, cs));
    expand_reads_kernel<<<(unsigned)((nb + 255) / 256), 256, 0, cs>>>(nb, stage.as<uint64_t>(), h->words, d_rec + r0 * ds, ds);
    c->launches++;
    if (h->n_with_n) {
        const uint32_t *lo = std::lower_bound(h->n_idx, h->n_idx + h->n_with_n, (uint32_t)std::min<uint64_t>(r0, 0xFFFFFFFFull));
        const uint32_t *hi = std::lower_bound(h->n_idx, h->n_idx + h->n_with_n, (uint32_t)std::min<uint64_t>(r0 + nb, 0xFFFFFFFFull));
        const size_t a = (size_t)(lo - h->n_idx), cnt = (size_t)(hi - lo);
        if (cnt) {
            c->d_nidx.ensure(h->n_with_n * 4 + 16); c->d_nmask.ensure(h->n_with_n * (size_t)h->words * 4 + 16);
            uint32_t *di = c->d_nidx.as<uint32_t>() + a, *dm = c->d_nmask.as<uint32_t>() + a * h->words;
            CK(cudaMemcpyAsync(di, lo, cnt * 4, cudaMemcpyHostToDevice, cs));
            CK(cudaMemcpyAsync(dm, h->n_mask + a * h->words, cnt * (size_t)h->words * 4, cudaMemcpyHostToDevice, cs));
            scatter_nmask_kernel<<<(unsigned)((cnt + 127) / 128), 128, 0, cs>>>((uint32_t)cnt, di, dm, h->words, d_rec, ds);
            c->launches++;
            bytes += cnt * (4 + (uint64_t)h->words * 4);
        }
    }
    return bytes;
}

// Allocates L's slab for an image of layout `lay` (library.cpp), points L.dev into it and uploads the feature token
// ranks.  The image itself arrives through copy_image.
static void place_library(nb200_ctx *c, DevLibrary &L, const ImageLayout &lay) {
    const HostLibrary &h = L.host;
    auto up = [&](DevBuf &b, const void *src, size_t bytes) {
        b.ensure(bytes ? bytes : 16);
        if (bytes) CK(cudaMemcpyAsync(b.p, src, bytes, cudaMemcpyHostToDevice, c->s_compute));
    };
    up(L.tok_end, h.tok_end.data(), h.tok_end.size() * 4);
    up(L.tok_comma, h.tok_comma.data(), h.tok_comma.size() * 4);
    if (h.has_index) {
        L.slab.ensure(lay.total + 256);
        L.slab_bytes = lay.total;
        const uint8_t *base = L.slab.as<uint8_t>();
        auto at = [&](int part) { return base + lay.off[part]; };
        L.table_bytes = lay.bytes[kPartTable];
        L.dev.table = reinterpret_cast<const uint4 *>(at(kPartTable));
        L.dev.n_buckets = (uint32_t)h.n_buckets;
        L.dev.dual = reinterpret_cast<const uint4 *>(at(kPartDual));
        L.dev.class_rec = reinterpret_cast<const uint4 *>(at(kPartClassRec));
        L.dev.ov_w = reinterpret_cast<const uint32_t *>(at(kPartOvW));
        L.dev.ov_b = reinterpret_cast<const uint32_t *>(at(kPartOvB));
        L.dev.ov_pre = reinterpret_cast<const uint32_t *>(at(kPartOvPre));
        L.dev.positions = reinterpret_cast<const uint32_t *>(at(kPartPositions));
        L.dev.ref_gstart = reinterpret_cast<const uint32_t *>(at(kPartRefGstart));
        L.dev.ref_feature = reinterpret_cast<const uint32_t *>(at(kPartRefFeature));
        L.dev.ref2bit = reinterpret_cast<const uint64_t *>(at(kPartRef2bit));
        L.dev.refN = reinterpret_cast<const uint32_t *>(at(kPartRefN));
        L.dev.n_refs = h.n_refs; L.dev.n_features = h.n_features; L.dev.n_words = h.n_words;
        L.dev.narrow_cap = kCap;
        if (const char *e = getenv("NB200_NARROW_CAP")) L.dev.narrow_cap = (uint32_t)std::min<long>(kCap, std::max<long>(0, atol(e)));   // tests: force the wide path
        if (const char *e = getenv("NB200_PROBE_WARP")) L.probe_warp = atol(e) != 0;
        L.dev.k = h.cfg.k; L.dev.identity = h.identity_features ? 1 : 0;
        L.dev.kmask = h.cfg.k == 32 ? ~0ull : ((1ull << (2 * h.cfg.k)) - 1);
        L.dev.kbits = h.cfg.k == 32 ? 0xFFFFFFFFull : ((1ull << h.cfg.k) - 1);
    }
    CK(cudaStreamSynchronize(c->s_compute));
}

// image bytes [offset, offset + len) into dst: from an index file or from a freshly built HostLibrary
using ImageFill = std::function<void(uint64_t offset, uint64_t len, uint8_t *dst)>;

// Copies one image of `total` bytes into the slab of Ls[d] on context cs[d], for every d: a pool of pinned staging
// buffers is filled chunk by chunk and each chunk goes to every device on its compute stream; a buffer is filled again
// once the copies out of it have completed on all devices.  Host memory is bounded by the pool, not by the image.
static void copy_image(const std::vector<nb200_ctx *> &cs, const std::vector<DevLibrary *> &Ls, uint64_t total, const ImageFill &fill) {
    constexpr uint64_t kChunk = 64ull << 20;
    constexpr uint64_t kBuffers = 4;
    struct Staging {
        void *p = nullptr;
        std::vector<Event> copied;              // per device
        ~Staging() { if (p) cudaFreeHost(p); }
    };
    std::vector<Staging> pool((size_t)std::min<uint64_t>(kBuffers, (total + kChunk - 1) / kChunk));
    auto drain = [&] { for (nb200_ctx *c : cs) { cudaSetDevice(c->device); cudaStreamSynchronize(c->s_compute); } };
    try {
        for (Staging &s : pool) {
            CK(cudaHostAlloc(&s.p, (size_t)std::min(kChunk, total), cudaHostAllocPortable));
            for (nb200_ctx *c : cs) {
                CK(cudaSetDevice(c->device));
                Event e;
                CK(cudaEventCreateWithFlags(&e.h, cudaEventDisableTiming));
                s.copied.push_back(std::move(e));
            }
        }
        uint64_t i = 0;
        for (uint64_t a = 0; a < total; a += kChunk, i++) {
            Staging &s = pool[i % pool.size()];
            const uint64_t n = std::min(kChunk, total - a);
            if (i >= pool.size()) for (Event &e : s.copied) CK(cudaEventSynchronize(e));
            fill(a, n, static_cast<uint8_t *>(s.p));
            for (size_t d = 0; d < cs.size(); d++) {
                CK(cudaSetDevice(cs[d]->device));
                CK(cudaMemcpyAsync(Ls[d]->slab.as<uint8_t>() + a, s.p, n, cudaMemcpyHostToDevice, cs[d]->s_compute));
                CK(cudaEventRecord(s.copied[d], cs[d]->s_compute));
            }
        }
        for (nb200_ctx *c : cs) { CK(cudaSetDevice(c->device)); CK(cudaStreamSynchronize(c->s_compute)); }
    } catch (...) {
        drain();                               // no copy may still read a staging buffer when the pool is freed
        throw;
    }
}

// Index-file check on the device: the checksum of checksum.hpp over the copy of the image the kernels will read.
// Grid-stride over 64-bit words, one atomicAdd per block.
__global__ void __launch_bounds__(256) image_checksum_kernel(const uint64_t *__restrict__ w, uint64_t n, unsigned long long *sum) {
    __shared__ unsigned long long part[8];
    unsigned long long s = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        s += image_word_sum(__ldg(w + i), i);
    for (int o = 16; o; o >>= 1) s += __shfl_down_sync(0xFFFFFFFFu, s, o);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int j = 1; j < 8; j++) s += part[j];
        atomicAdd(sum, s);
    }
}

// Runs image_checksum_kernel on every device side by side; throws when a device's copy differs from `want`.
static void check_image_sums(const std::vector<nb200_ctx *> &cs, const std::vector<DevLibrary *> &Ls, uint64_t want, const std::string &path,
                             float *kernel_ms) {
    std::vector<DevBuf> sum(cs.size());
    std::vector<Event> t0(cs.size()), t1(cs.size());
    std::vector<unsigned long long> got(cs.size(), 0);
    for (size_t d = 0; d < cs.size(); d++) {
        nb200_ctx *c = cs[d];
        CK(cudaSetDevice(c->device));
        CK(cudaEventCreate(&t0[d].h)); CK(cudaEventCreate(&t1[d].h));
        sum[d].ensure(8);
        CK(cudaMemsetAsync(sum[d].p, 0, 8, c->s_compute));
        CK(cudaEventRecord(t0[d], c->s_compute));
        image_checksum_kernel<<<(unsigned)c->sm_count * 8, 256, 0, c->s_compute>>>(Ls[d]->slab.as<uint64_t>(), Ls[d]->slab_bytes / 8,
                                                                                  sum[d].as<unsigned long long>());
        CK(cudaGetLastError());
        CK(cudaEventRecord(t1[d], c->s_compute));
        c->launches++;
        CK(cudaMemcpyAsync(&got[d], sum[d].p, 8, cudaMemcpyDeviceToHost, c->s_compute));
    }
    *kernel_ms = 0.0f;
    for (size_t d = 0; d < cs.size(); d++) {
        CK(cudaSetDevice(cs[d]->device));
        CK(cudaStreamSynchronize(cs[d]->s_compute));
        float ms = 0.0f;
        CK(cudaEventElapsedTime(&ms, t0[d], t1[d]));
        *kernel_ms = std::max(*kernel_ms, ms);
        sum[d].release();
    }
    for (size_t d = 0; d < cs.size(); d++)
        if (got[d] != want)
            throw std::runtime_error("index file " + path + " is damaged: the device image on GPU " + std::to_string(cs[d]->device) +
                                     " fails its checksum");
}

// One library onto every context of `cs`, under the same id on each (they hold the same libraries): `meta` is the library
// without its images, `fill` produces the image of `lay`, copied once to all devices.  With `want_sum` (an index file)
// each device checks its copy; a failure leaves every context as it was.
static void install_library(const std::vector<nb200_ctx *> &cs, const HostLibrary &meta, const ImageLayout &lay, const ImageFill &fill,
                            const uint64_t *want_sum, const std::string &path, double host_s, int32_t *lib_id) {
    std::vector<std::unique_ptr<DevLibrary>> Ls;
    std::vector<DevLibrary *> raw;
    auto t0 = std::chrono::steady_clock::now();
    float sum_ms = 0.0f;
    try {
        for (nb200_ctx *c : cs) {
            CK(cudaSetDevice(c->device));
            Ls.push_back(std::make_unique<DevLibrary>());
            Ls.back()->host = library_meta(meta);
            raw.push_back(Ls.back().get());
            place_library(c, *Ls.back(), lay);
        }
        if (meta.has_index) {
            copy_image(cs, raw, lay.total, fill);
            if (want_sum) check_image_sums(cs, raw, *want_sum, path, &sum_ms);
        }
    } catch (...) {
        for (size_t d = 0; d < Ls.size(); d++) { cudaSetDevice(cs[d]->device); Ls[d].reset(); }   // frees each slab on its own device
        throw;
    }
    if (getenv("NB200_TRACE") && meta.has_index)
        fprintf(stderr, "[nb200 trace] library %s: %s %.3f s, image %.1f MB to %zu GPUs %.3f s, device checksum %.3f ms\n", path.c_str(),
                want_sum ? "index read" : "index built", host_s, lay.total / 1e6, cs.size(),
                std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count(), sum_ms);
    for (size_t d = 0; d < cs.size(); d++) {
        cs[d]->libs.push_back(std::move(Ls[d]));
        if (d == 0 && lib_id) *lib_id = (int32_t)cs[d]->libs.size() - 1;
    }
}

// From a library JSON (built on the host) or an index file (told apart by its magic bytes, not its extension): the
// library loaded onto every context of `cs`.  k <= 0: the index's own k, or 20 for a JSON.
static void load_library_path(const std::vector<nb200_ctx *> &cs, const char *path, const char *strand_filter, int32_t k, int host_threads,
                              int32_t *lib_id) {
    if (!path) throw std::runtime_error("library path is null");
    const int sf = parse_strand_filter(strand_filter);
    if (sf < 0) throw std::runtime_error(std::string("unknown --strand_filter value: ") + strand_filter);
    const auto t0 = std::chrono::steady_clock::now();
    auto since = [&] { return std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count(); };
    if (is_index_file(path)) {
        IndexFile f;
        HostLibrary meta;
        open_index_file(path, f, meta);
        if (k > 0 && k != meta.cfg.k)
            throw std::runtime_error(std::string("index file ") + path + " was built with k = " + std::to_string(meta.cfg.k) +
                                     "; the call asks for k = " + std::to_string(k));
        meta.cfg.strand_filter = sf;
        const uint64_t want = f.h.sec[kSecImage].sum;
        install_library(cs, meta, image_layout(f.h.part_bytes), [&](uint64_t a, uint64_t n, uint8_t *dst) { f.read_image(a, n, dst); },
                        &want, path, since(), lib_id);
        return;
    }
    std::vector<std::string> names, seqs, feats;
    nb200_config cfg{};
    parse_library_json(path, names, seqs, feats, cfg);
    cfg.k = k > 0 ? k : 20;
    cfg.strand_filter = sf;
    HostLibrary h;
    build_library(names, seqs, feats, cfg, host_threads, h, getenv("NB200_VERIFY_TABLE") != nullptr);
    const ImageLayout lay = image_layout(h);
    install_library(cs, h, lay, [&](uint64_t a, uint64_t n, uint8_t *dst) { image_fill(h, lay, a, n, dst); }, nullptr, path, since(), lib_id);
}

// Keep the index resident in L2 while reads and per-read outputs stream through it: persisting
// access-policy window over the slab on the compute stream (hit ratio scaled to the set-aside).
static void pin_index_in_l2(nb200_ctx *c, const DevLibrary &L) {
    if (!L.host.has_index || c->l2_persist_max == 0 || c->l2_window_lib == &L) return;
    cudaStreamAttrValue v{};
    size_t win = std::min<size_t>(L.slab_bytes, (size_t)c->l2_window_max);
    v.accessPolicyWindow.base_ptr = L.slab.p;
    v.accessPolicyWindow.num_bytes = win;
    v.accessPolicyWindow.hitRatio = (float)std::min(1.0, (double)c->l2_persist_max / (double)std::max<size_t>(win, 1));
    v.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
    v.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
    if (cudaStreamSetAttribute(c->s_compute, cudaStreamAttributeAccessPolicyWindow, &v) != cudaSuccess) cudaGetLastError();
    if (cudaStreamSetAttribute(c->s_tail, cudaStreamAttributeAccessPolicyWindow, &v) != cudaSuccess) cudaGetLastError();
    c->l2_window_lib = &L;
}

constexpr int kMinScoreLen = 513;     // read lengths 0..512 (16 packed words)

// CallParams for a library + its score_percent table: min_score[len] = smallest s with !((double)s / (double)len <
// score_percent), evaluated with the expression the SPEC (and the oracle) uses, so `score < min_score[len]` is that test.
static CallParams call_params(nb200_ctx *c, DevLibrary &L) {
    const nb200_config &cfg = L.host.cfg;
    CallParams p;
    p.score_threshold = cfg.score_threshold; p.score_filter = cfg.score_filter; p.num_mismatches = cfg.num_mismatches;
    p.discard_multiple_matches = cfg.discard_multiple_matches; p.intersect_level = cfg.intersect_level;
    p.discard_multi_hits = cfg.discard_multi_hits; p.require_valid_pair = cfg.require_valid_pair;
    p.max_hits = cfg.max_hits_to_report; p.strand_filter = cfg.strand_filter;
    const double sp = cfg.score_percent;
    if (!L.min_score_ok || memcmp(&L.min_score_for, &sp, sizeof sp) != 0) {
        uint16_t tab[kMinScoreLen];
        for (int len = 0; len < kMinScoreLen; len++) {
            int lo = 0, hi = 65535;                               // the test is monotone in s (correctly rounded division)
            if ((double)hi / (double)len < sp) { tab[len] = 65535; continue; }     // nothing passes (scores never reach 65535)
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if ((double)mid / (double)len < sp) lo = mid + 1; else hi = mid;
            }
            tab[len] = (uint16_t)lo;
        }
        CK(cudaDeviceSynchronize());                              // no kernel may still read the old table
        L.min_score.ensure(sizeof tab);
        CK(cudaMemcpy(L.min_score.p, tab, sizeof tab, cudaMemcpyHostToDevice));
        L.min_score_for = sp; L.min_score_ok = true;
    }
    p.min_score = L.min_score.as<uint16_t>();
    return p;
}

// One batch.  Probe + wide-read kernels on s_compute; fingerprint / dedupe / Smith-Waterman / deferred calling on the
// high-priority s_tail, so that they run beside the NEXT batch's probe (they are latency bound, the probe is issue
// bound).  Per-batch state is double-buffered: a slot is reused only after its tail has finished.
static inline unsigned nblk(uint64_t n, unsigned t) { return (unsigned)((n + t - 1) / t); }

struct BatchIO {                 // where a batch reads its reads and writes its per-read outputs (entry 0 = read `read0`)
    ReadsDev r1, r2;
    nb200_read_result *res;
    int32_t *feats;
    uint16_t *nf;
};

static void launch_batch(nb200_ctx *c, const DevLibrary &L, const CallParams &cp, const BatchIO &io, uint64_t read0, uint64_t nb, int n_mates,
                         int slot, cudaEvent_t e_start, cudaEvent_t e_probe, cudaEvent_t e_tail0, cudaEvent_t e_sw, cudaEvent_t e_call,
                         cudaEvent_t e_pk = nullptr) {
    nb200_ctx::BatchBuf &B = c->bb[slot];
    cudaStream_t sp = c->s_compute, st = c->overlap ? c->s_tail : c->s_compute;
    if (B.busy && c->overlap) CK(cudaStreamWaitEvent(sp, B.tail_done, 0));
    if (e_start) CK(cudaEventRecord(e_start, sp));
    const unsigned pthreads = kProbeWarps * 32;
    const unsigned blocks = (unsigned)((nb * 32 + pthreads - 1) / pthreads);
    nb200_read_result *res = io.res;
    int32_t *feats = io.feats;
    uint16_t *nf = io.nf;
    const ReadsDev &r1 = io.r1, &r2 = io.r2;
    RoRec *ro = B.ro.as<RoRec>();
    uint32_t *roB = B.roB.as<uint32_t>(), *deferred = B.deferred.as<uint32_t>(), *wide_list = B.wide_list.as<uint32_t>();
    uint32_t *warp_list = B.warp_list.as<uint32_t>();
    SwItem *items = B.items.as<SwItem>();
    OriSum *sums = B.sums.as<OriSum>();
    uint32_t *slow_list = B.slow_list.as<uint32_t>(), *setup_list = B.setup_list.as<uint32_t>();
#define NB200_PROBE(NM, ST) probe_kernel<NM, ST><<<blocks, pthreads, 0, sp>>>(L.dev, r1, r2, read0, nb, sums, roB, wide_list, B.ctr)
    // single-end: one thread per read, then the warp form on the reads it could not keep in registers
#define NB200_PROBE_THREAD(ST)                                                                                                \
    probe_thread_kernel<ST><<<nblk(nb, kProbeThreads), kProbeThreads, 0, sp>>>(L.dev, r1, read0, nb, sums, warp_list, B.ctr); \
    probe_list_kernel<ST><<<c->sm_count * kProbeListBlocks, pthreads, 0, sp>>>(L.dev, r1, read0, warp_list, sums, roB, wide_list, B.ctr)
    if (n_mates == 2) { if (c->stats) NB200_PROBE(2, true); else NB200_PROBE(2, false); }
    else if (L.probe_warp) { if (c->stats) NB200_PROBE(1, true); else NB200_PROBE(1, false); }
    else { if (c->stats) { NB200_PROBE_THREAD(true); } else { NB200_PROBE_THREAD(false); } }
#undef NB200_PROBE_THREAD
#undef NB200_PROBE
    if (e_pk) CK(cudaEventRecord(e_pk, sp));          // the probe kernels alone (the roofline's kernel), before the calling kernels
    // reads whose narrowest class is wider than the shared-memory lists (rare): generic path on global scratch
    wide_kernel<<<kWideBlocks, 128, 0, sp>>>(L.dev, cp, r1, r2, read0, n_mates, wide_list, c->wide_scratch.as<uint32_t>(),
                                             c->wide_v.as<uint32_t>(), res, feats, nf, B.ctr);
    // score / filter / feature call: one thread per read; the reads that need alignment (or carry wide sets): one warp each
    const size_t fast_smem = (size_t)kFastThreads * (10 + cp.max_hits) * 4;      // per-read outputs staged for coalesced stores
    if (fast_smem > 48 * 1024) {      // max_hits_to_report beyond 38: more dynamic shared memory than the default limit
        CK(cudaFuncSetAttribute(call_fast_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fast_smem));
        CK(cudaFuncSetAttribute(call_fast_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fast_smem));
    }
    if (n_mates == 2) {
        call_fast_kernel<2><<<nblk(nb, kFastThreads), kFastThreads, fast_smem, sp>>>(L.dev, cp, sums, (uint32_t)nb, slow_list, setup_list, res, feats, nf, B.ctr);
        sw_setup_kernel<2><<<c->sm_count * 8, 128, 0, sp>>>(L.dev, r1, r2, read0, sums, setup_list, ro, roB, deferred, items, c->items_cap, B.ctr);
        call_slow_kernel<2><<<c->sm_count * 2, 128, 0, sp>>>(L.dev, cp, r1, r2, read0, sums, slow_list, ro, roB, deferred, items, c->items_cap,
                                                             res, feats, nf, B.ctr);
    } else {
        call_fast_kernel<1><<<nblk(nb, kFastThreads), kFastThreads, fast_smem, sp>>>(L.dev, cp, sums, (uint32_t)nb, slow_list, setup_list, res, feats, nf, B.ctr);
        sw_setup_kernel<1><<<c->sm_count * 8, 128, 0, sp>>>(L.dev, r1, r2, read0, sums, setup_list, ro, roB, deferred, items, c->items_cap, B.ctr);
        call_slow_kernel<1><<<c->sm_count * 2, 128, 0, sp>>>(L.dev, cp, r1, r2, read0, sums, slow_list, ro, roB, deferred, items, c->items_cap,
                                                             res, feats, nf, B.ctr);
    }
    if (st != sp) { CK(cudaEventRecord(B.probe_done, sp)); CK(cudaStreamWaitEvent(st, B.probe_done, 0)); }
    if (e_probe) CK(cudaEventRecord(e_probe, sp));
    if (e_tail0) CK(cudaEventRecord(e_tail0, st));
    window_hash_kernel<<<c->sm_count * 8, 256, 0, st>>>(L.dev, items, c->items_cap, B.ctr);
    dedupe_kernel<<<c->sm_count * 8, 256, 0, st>>>(L.dev, items, c->items_cap, B.sw_rep.as<uint32_t>(), B.sw_pairs.as<uint32_t>(), B.ctr);
    sw_kernel<<<c->sm_count * 8, 128, 0, st>>>(L.dev, r1, r2, read0, n_mates, deferred, items, c->items_cap,
                                               B.sw_pairs.as<uint32_t>(), B.ctr);
    if (e_sw) CK(cudaEventRecord(e_sw, st));
    if (n_mates == 2)
        call_deferred_thread_kernel<2><<<c->sm_count * 8, 128, 0, st>>>(L.dev, cp, ro, roB, deferred, items, B.sw_rep.as<uint32_t>(), c->items_cap,
                                                                       res, feats, nf, slow_list, B.ctr);
    else
        call_deferred_thread_kernel<1><<<c->sm_count * 8, 128, 0, st>>>(L.dev, cp, ro, roB, deferred, items, B.sw_rep.as<uint32_t>(), c->items_cap,
                                                                       res, feats, nf, slow_list, B.ctr);
    if (n_mates == 2)
        call_deferred_kernel<2><<<c->sm_count * 2, 256, 0, st>>>(L.dev, cp, ro, roB, deferred, items, B.sw_rep.as<uint32_t>(), c->items_cap,
                                                                 res, feats, nf, slow_list, B.ctr);
    else
        call_deferred_kernel<1><<<c->sm_count * 2, 256, 0, st>>>(L.dev, cp, ro, roB, deferred, items, B.sw_rep.as<uint32_t>(), c->items_cap,
                                                                 res, feats, nf, slow_list, B.ctr);
    end_batch_kernel<<<1, 1, 0, st>>>(B.ctr);
    if (e_call) CK(cudaEventRecord(e_call, st));
    CK(cudaEventRecord(B.tail_done, st));
    B.busy = true;
    c->launches += (n_mates == 1 && !L.probe_warp) ? 12 : 11;
}

static void cub_sort32(nb200_ctx *c, const uint32_t *kin, uint32_t *kout, const uint32_t *vin, uint32_t *vout, uint32_t m, int bits) {
    size_t bytes = 0;
    CK(cub::DeviceRadixSort::SortPairs(nullptr, bytes, kin, kout, vin, vout, (int)m, 0, bits, c->s_compute));
    c->cub_tmp.ensure(bytes);
    CK(cub::DeviceRadixSort::SortPairs(c->cub_tmp.p, bytes, kin, kout, vin, vout, (int)m, 0, bits, c->s_compute));
}
static void cub_sort64(nb200_ctx *c, const uint64_t *kin, uint64_t *kout, const uint32_t *vin, uint32_t *vout, uint32_t m, int bits) {
    size_t bytes = 0;
    CK(cub::DeviceRadixSort::SortPairs(nullptr, bytes, kin, kout, vin, vout, (int)m, 0, bits, c->s_compute));
    c->cub_tmp.ensure(bytes);
    CK(cub::DeviceRadixSort::SortPairs(c->cub_tmp.p, bytes, kin, kout, vin, vout, (int)m, 0, bits, c->s_compute));
}
// indices of set flags -> out; returns the count (one host sync)
static uint32_t cub_select(nb200_ctx *c, const uint8_t *flag, uint32_t *out, uint32_t n) {
    size_t bytes = 0;
    thrust::counting_iterator<uint32_t> it(0);
    c->num.ensure(64);
    CK(cub::DeviceSelect::Flagged(nullptr, bytes, it, flag, out, c->num.as<uint32_t>(), (int)n, c->s_compute));
    c->cub_tmp.ensure(bytes);
    CK(cub::DeviceSelect::Flagged(c->cub_tmp.p, bytes, it, flag, out, c->num.as<uint32_t>(), (int)n, c->s_compute));
    uint32_t h = 0;
    CK(cudaMemcpyAsync(&h, c->num.p, 4, cudaMemcpyDeviceToHost, c->s_compute));
    CK(cudaStreamSynchronize(c->s_compute));
    c->timing.d2h_bytes += 4;
    return h;
}
// indices of set flags -> out, the count -> *d_count (device); no host sync
static void cub_select_async(nb200_ctx *c, const uint8_t *flag, uint32_t *out, uint32_t n, uint32_t *d_count) {
    size_t bytes = 0;
    thrust::counting_iterator<uint32_t> it(0);
    CK(cub::DeviceSelect::Flagged(nullptr, bytes, it, flag, out, d_count, (int)n, c->s_compute));
    c->cub_tmp.ensure(bytes);
    CK(cub::DeviceSelect::Flagged(c->cub_tmp.p, bytes, it, flag, out, d_count, (int)n, c->s_compute));
}
// the aggregation's device scalars (c->num): 0 groups, 1 largest group, 2 UMIs for the general kernel, 3 distinct lists,
// 4 ids of the table, 5 UMIs with a result, 6 table rows, 7 selected rows, 8 longest selected row, 9 UMIs corrected
enum { DV_GROUPS = 0, DV_MAXGROUP, DV_GENERAL, DV_LISTS, DV_IDS, DV_LIVE, DV_ROWS, DV_SELECTED, DV_MAXLEN, DV_CORRECTED, DV_COUNT };
static void fetch_scalars(nb200_ctx *c, uint32_t *h) {           // ONE host sync for all of them
    CK(cudaMemcpyAsync(h, c->num.p, DV_COUNT * 4, cudaMemcpyDeviceToHost, c->s_compute));
    CK(cudaStreamSynchronize(c->s_compute));
    c->timing.d2h_bytes += DV_COUNT * 4;
}
static void excl_scan_u32(nb200_ctx *c, const uint32_t *in, uint32_t *out, uint32_t n) {
    size_t bytes = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, bytes, in, out, (int)n, c->s_compute));
    c->cub_tmp.ensure(bytes);
    CK(cub::DeviceScan::ExclusiveSum(c->cub_tmp.p, bytes, in, out, (int)n, c->s_compute));
}
static void incl_scan_u32(nb200_ctx *c, const uint32_t *in, uint32_t *out, uint32_t n) {
    size_t bytes = 0;
    CK(cub::DeviceScan::InclusiveSum(nullptr, bytes, in, out, (int)n, c->s_compute));
    c->cub_tmp.ensure(bytes);
    CK(cub::DeviceScan::InclusiveSum(c->cub_tmp.p, bytes, in, out, (int)n, c->s_compute));
}

// LSD radix over token-rank columns: afterwards permA orders the listed rows by the byte order
// of their comma-joined feature strings (stable).
static void sort_by_feature_string(nb200_ctx *c, const DevLibrary &L, uint32_t m, const Rows &rows, uint32_t max_nf) {
    int bits = 1;
    while ((1ull << bits) < 2ull * L.host.n_features + 2) bits++;
    c->k32A.ensure((size_t)m * 4); c->k32B.ensure((size_t)m * 4); c->permB.ensure((size_t)m * 4);
    const int per_key = std::max(1, 32 / bits);          // token columns per 32-bit radix key
    for (int hi = (int)max_nf; hi > 0; hi -= per_key) {   // LSD: last group of columns first
        const int p0 = std::max(0, hi - per_key), cols = hi - p0;
        gather_tok_kernel<<<nblk(m, 256), 256, 0, c->s_compute>>>(m, c->permA.as<uint32_t>(), rows, (uint32_t)p0, (uint32_t)cols,
                                                                    (uint32_t)bits, L.tok_end.as<uint32_t>(), L.tok_comma.as<uint32_t>(),
                                                                    c->k32A.as<uint32_t>());
        c->launches++;
        cub_sort32(c, c->k32A.as<uint32_t>(), c->k32B.as<uint32_t>(), c->permA.as<uint32_t>(), c->permB.as<uint32_t>(), m, bits * cols);
        std::swap(c->permA, c->permB);
    }
}

// the count table lives in pinned host memory owned by the context
static void ensure_host_table(nb200_ctx *c, size_t nrows, size_t ids) {
    auto grow = [](PinnedBuf<uint32_t> &b, size_t n) { if (n + 1 > b.cap) b.ensure(n + n / 4 + 1024); };
    grow(c->h_cell, nrows); grow(c->h_count, nrows); grow(c->h_off, nrows);
    grow(c->h_ids, ids);
}

static int bits_for(uint64_t n) { int b = 1; while ((1ull << b) < n) b++; return b; }

// UMI correction (DESIGN.md §2.12) over the m selected rows (permA, input order): rows counted per key in a table sized
// from m, every key's target found from those counts, each row's key rewritten to its target's.  Returns the rewritten
// keys, indexed like d_key (only the selected rows' entries are written); the number of keys corrected goes to
// dv[DV_CORRECTED].
static const uint64_t *correct_umis(nb200_ctx *c, uint64_t n, const uint64_t *d_key, uint32_t m, uint32_t *dv) {
    uint32_t tsize = 1024;
    while (tsize < 2ull * m && tsize < (1u << 31)) tsize <<= 1;      // load factor <= 0.5 (m < 2^31 keeps a slot free)
    c->k64A.ensure((size_t)m * 8); c->umi_table.ensure((size_t)tsize * sizeof(UmiSlot)); c->umi_key.ensure(n * 8);
    UmiSlot *t = c->umi_table.as<UmiSlot>();
    CK(cudaMemsetAsync(t, 0, (size_t)tsize * sizeof(UmiSlot), c->s_compute));
    gather_key64_kernel<<<nblk(m, 256), 256, 0, c->s_compute>>>(m, c->permA.as<uint32_t>(), d_key, c->k64A.as<uint64_t>());
    umi_count_kernel<<<nblk(m, 256), 256, 0, c->s_compute>>>(m, c->k64A.as<uint64_t>(), t, tsize - 1);
    umi_correct_kernel<<<nblk(tsize, 256), 256, 0, c->s_compute>>>(tsize, t, tsize - 1, dv + DV_CORRECTED);
    umi_rewrite_kernel<<<nblk(m, 256), 256, 0, c->s_compute>>>(m, c->permA.as<uint32_t>(), c->k64A.as<uint64_t>(), t, tsize - 1,
                                                                c->umi_key.as<uint64_t>());
    c->launches += 4;
    return c->umi_key.as<uint64_t>();
}

// A6 (nimble/__main__.py:234-293).  Inputs resident on device; fills ctx->o_* host vectors.
// rows: padded or CSR (agg.cuh); max_nf_hint: longest row if known (0: stride); ids_bound: upper bound of the names of
// all rows together (sizes nothing but a sanity check; the pools are sized from the device-side total).
// umi_flags: NB200_UMI_NO_THRESHOLD, NB200_UMI_CORRECT (keyed rows only; bulk data has no UMIs).
static void aggregate(nb200_ctx *c, const DevLibrary &L, uint64_t n, const uint64_t *d_key, const Rows &rows,
                      const double *d_score, uint32_t max_nf_hint, double threshold, int umi_flags, nb200_counts *counts) {
    const int disable = umi_flags & NB200_UMI_NO_THRESHOLD;
    counts->n_rows = 0; counts->dropped_empty = 0; counts->n_called = 0; counts->n_umis = 0;
    c->dev_rows = 0; c->dev_ids = 0;
    c->umis_corrected = 0;
    auto host_rows = [&](size_t nrows, size_t ids) { ensure_host_table(c, nrows, ids); };
    if (c->fetch_started) { CK(cudaStreamSynchronize(c->s_copy[1])); c->fetch_started = false; }      // (a fetch nobody waited for)
    c->fetch_pending = false;
    host_rows(0, 0);
    c->h_off.p[0] = 0;
    auto finish = [&]() {
        counts->cell = c->h_cell.p; counts->count = c->h_count.p;
        counts->feat_off = c->h_off.p; counts->feat_ids = c->h_ids.p;
    };
    if (n == 0 || n > 0x7FFFFFF0ull) { if (n) throw LimitError("more than 2^31 rows in one call (CUB item counts are int)"); finish(); return; }
    const bool bulk = d_key == nullptr;
    uint32_t hv[DV_COUNT];
    c->num.ensure(64);
    uint32_t *dv = c->num.as<uint32_t>();
    CK(cudaMemsetAsync(dv, 0, DV_COUNT * 4, c->s_compute));
    c->flag.ensure(n); c->permA.ensure(n * 4);
    mark_rows_kernel<<<nblk(n, 256), 256, 0, c->s_compute>>>(n, d_key, rows, d_score, c->flag.as<uint8_t>(), dv + DV_MAXLEN);
    c->launches++;
    cub_select_async(c, c->flag.as<uint8_t>(), c->permA.as<uint32_t>(), (uint32_t)n, dv + DV_SELECTED);
    fetch_scalars(c, hv);
    const uint32_t m = hv[DV_SELECTED];
    counts->n_called = m;
    if (m == 0) { finish(); return; }
    (void)max_nf_hint;
    const uint32_t max_nf = std::max(1u, hv[DV_MAXLEN]);      // token columns the feature-string sorts have to cover
    uint32_t G = 0;
    c->row_n.ensure(((size_t)m + 1) * 4); c->row_off.ensure(((size_t)m + 1) * 4);
    UmiOut uo{};
    const uint32_t *d_gstart = nullptr;              // UMI g -> its first sorted row (nullptr: bulk, UMI g is sorted row g)
    if (!bulk) {
        // rows -> (key, feature-string order, input order).  The key sort is stable on the input order; the feature
        // strings only have to be ordered INSIDE each (cell, umi) group, which is a handful of rows: a per-group
        // insertion sort replaces a global LSD sort over every token column of every row.
        c->k64A.ensure((size_t)m * 8); c->k64B.ensure((size_t)m * 8); c->permB.ensure((size_t)m * 4);
        c->head.ensure(m); c->gstart.ensure((size_t)m * 4);
        if (umi_flags & NB200_UMI_CORRECT) d_key = correct_umis(c, n, d_key, m, dv);
        auto sort_by_key = [&]() {
            gather_key64_kernel<<<nblk(m, 256), 256, 0, c->s_compute>>>(m, c->permA.as<uint32_t>(), d_key, c->k64A.as<uint64_t>());
            c->launches++;
            cub_sort64(c, c->k64A.as<uint64_t>(), c->k64B.as<uint64_t>(), c->permA.as<uint32_t>(), c->permB.as<uint32_t>(), m, 64);
            std::swap(c->permA, c->permB);
        };
        sort_by_key();
        key_heads_kernel<<<nblk(m + 1, 256), 256, 0, c->s_compute>>>(m, c->k64B.as<uint64_t>(), c->permA.as<uint32_t>(), rows,
                                                                      c->head.as<uint8_t>(), c->row_n.as<uint32_t>());
        cub_select_async(c, c->head.as<uint8_t>(), c->gstart.as<uint32_t>(), m, dv + DV_GROUPS);
        max_group_kernel<<<nblk(m, 256), 256, 0, c->s_compute>>>(dv, c->gstart.as<uint32_t>(), m, dv + DV_MAXGROUP);
        // pools: exclusive scan of the names per sorted row (a group's total does not depend on the order inside it)
        excl_scan_u32(c, c->row_n.as<uint32_t>(), c->row_off.as<uint32_t>(), m + 1);
        CK(cudaMemcpyAsync(dv + DV_IDS, c->row_off.as<uint32_t>() + m, 4, cudaMemcpyDeviceToDevice, c->s_compute));
        c->launches += 3;
        fetch_scalars(c, hv);
        G = hv[DV_GROUPS];
        const uint32_t T = hv[DV_IDS];
        counts->n_umis = G;
        c->umis_corrected = hv[DV_CORRECTED];
        if (hv[DV_MAXGROUP] <= kLocalSortMax) {
            group_sort_kernel<<<nblk(G, 128), 128, 0, c->s_compute>>>(G, c->gstart.as<uint32_t>(), m, c->permA.as<uint32_t>(), rows,
                                                                       L.tok_end.as<uint32_t>(), L.tok_comma.as<uint32_t>());
            c->launches++;
        } else {
            // a very large group (e.g. data without real UMIs): global stable token sort, then the key sort again
            sort_by_feature_string(c, L, m, rows, max_nf);
            sort_by_key();
        }
        c->u_cell.ensure((size_t)G * 4); c->u_n.ensure((size_t)G * 2); c->u_list.ensure((size_t)T * 4 + 16);
        c->slow.ensure((size_t)G * 4);
        c->s_rep.ensure((size_t)m * 4); c->s_S.ensure((size_t)m * 8);
        c->s_U.ensure((size_t)T * 4 + 16); c->s_fs.ensure((size_t)T * 8 + 16); c->s_fc.ensure((size_t)T * 8 + 16);
        c->s_flags.ensure((size_t)T + 16);
        uo = UmiOut{c->u_cell.as<uint32_t>(), c->u_n.as<uint16_t>(), c->u_list.as<int32_t>()};
        UmiScratch sc{c->row_off.as<uint32_t>(), c->s_rep.as<uint32_t>(), c->s_S.as<double>(), c->s_U.as<uint32_t>(),
                      c->s_fs.as<double>(), c->s_fc.as<double>(), c->s_flags.as<uint8_t>()};
        umi_simple_kernel<<<nblk(G, 128), 128, 0, c->s_compute>>>(G, c->gstart.as<uint32_t>(), m, c->permA.as<uint32_t>(),
                                                                   c->k64B.as<uint64_t>(), rows, d_score, threshold, disable,
                                                                   c->row_off.as<uint32_t>(), uo, c->slow.as<uint32_t>(), dv);
        umi_general_kernel<<<c->sm_count * 16, 128, 0, c->s_compute>>>(c->slow.as<uint32_t>(), dv, G, c->gstart.as<uint32_t>(), m,
                                                                       c->permA.as<uint32_t>(), c->k64B.as<uint64_t>(), rows, d_score,
                                                                       threshold, disable, sc, uo, c->d_ctr.as<Counters>());
        c->launches += 2;
        d_gstart = c->gstart.as<uint32_t>();
    } else {
        G = m;
        row_len_kernel<<<nblk(m + 1, 256), 256, 0, c->s_compute>>>(m, c->permA.as<uint32_t>(), rows, c->row_n.as<uint32_t>());
        excl_scan_u32(c, c->row_n.as<uint32_t>(), c->row_off.as<uint32_t>(), m + 1);
        CK(cudaMemcpyAsync(dv + DV_IDS, c->row_off.as<uint32_t>() + m, 4, cudaMemcpyDeviceToDevice, c->s_compute));
        fetch_scalars(c, hv);
        const uint32_t T = hv[DV_IDS];
        c->u_cell.ensure((size_t)G * 4); c->u_n.ensure((size_t)G * 2); c->u_list.ensure((size_t)T * 4 + 16);
        uo = UmiOut{c->u_cell.as<uint32_t>(), c->u_n.as<uint16_t>(), c->u_list.as<int32_t>()};
        bulk_rows_kernel<<<nblk(m, 256), 256, 0, c->s_compute>>>(m, c->permA.as<uint32_t>(), rows, c->row_off.as<uint32_t>(), uo);
        c->launches += 3;
    }
    // ---- second stage: count UMIs per (cell, feature list) -------------------------------------
    // result lists -> representatives (hash table), distinct lists ranked by feature string, ONE sort on (cell ordinal, rank)
    const Rows lists{uo.list, c->row_off.as<uint32_t>(), d_gstart, uo.n, 0};
    uint32_t tsize = 1024;
    while (tsize < 2ull * G && tsize < (1u << 31)) tsize <<= 1;
    c->htable.ensure((size_t)tsize * 4); c->rep_of.ensure((size_t)G * 4); c->is_rep.ensure(G);
    c->cell_ord.ensure((size_t)G * 4); c->rank_of.ensure((size_t)G * 4); c->k32A.ensure((size_t)G * 4);
    CK(cudaMemsetAsync(c->htable.p, 0, (size_t)tsize * 4, c->s_compute));
    CK(cudaMemsetAsync(dv + DV_IDS, 0, 4, c->s_compute));
    dedupe_lists_kernel<<<nblk(G, 256), 256, 0, c->s_compute>>>(G, lists, c->htable.as<uint32_t>(), tsize - 1, c->rep_of.as<uint32_t>(),
                                                                 c->is_rep.as<uint8_t>());
    c->permA.ensure((size_t)G * 4);
    cub_select_async(c, c->is_rep.as<uint8_t>(), c->permA.as<uint32_t>(), G, dv + DV_LISTS);
    cell_heads_kernel<<<nblk(G, 256), 256, 0, c->s_compute>>>(G, uo.cell, c->k32A.as<uint32_t>());
    incl_scan_u32(c, c->k32A.as<uint32_t>(), c->cell_ord.as<uint32_t>(), G);
    CK(cudaMemcpyAsync(dv + DV_ROWS, c->cell_ord.as<uint32_t>() + (G - 1), 4, cudaMemcpyDeviceToDevice, c->s_compute));
    c->launches += 4;
    fetch_scalars(c, hv);
    const uint32_t D = hv[DV_LISTS], n_cells = hv[DV_ROWS] + 1;
    if (D == 0) { finish(); return; }
    sort_by_feature_string(c, L, D, lists, max_nf);        // permA: the representatives in feature-string order
    scatter_rank_kernel<<<nblk(D, 256), 256, 0, c->s_compute>>>(D, c->permA.as<uint32_t>(), c->rank_of.as<uint32_t>());
    const int rank_bits = bits_for(D), cell_bits = bits_for(n_cells);
    const uint64_t sentinel = 1ull << (rank_bits + cell_bits);
    c->k64A.ensure((size_t)G * 8); c->k64B.ensure((size_t)G * 8); c->permA.ensure((size_t)G * 4); c->permB.ensure((size_t)G * 4);
    umi_keys_kernel<<<nblk(G, 256), 256, 0, c->s_compute>>>(G, c->cell_ord.as<uint32_t>(), c->rep_of.as<uint32_t>(), c->rank_of.as<uint32_t>(),
                                                             (uint32_t)rank_bits, sentinel, c->k64A.as<uint64_t>(), c->permA.as<uint32_t>());
    cub_sort64(c, c->k64A.as<uint64_t>(), c->k64B.as<uint64_t>(), c->permA.as<uint32_t>(), c->permB.as<uint32_t>(), G, rank_bits + cell_bits + 1);
    std::swap(c->permA, c->permB);
    c->head.ensure(G); c->gstart2.ensure((size_t)G * 4);
    run_heads_kernel<<<nblk(G, 256), 256, 0, c->s_compute>>>(G, c->k64B.as<uint64_t>(), c->permA.as<uint32_t>(), sentinel, uo.n,
                                                              c->head.as<uint8_t>(), dv);
    cub_select_async(c, c->head.as<uint8_t>(), c->gstart2.as<uint32_t>(), G, dv + DV_ROWS);
    c->launches += 4;
    fetch_scalars(c, hv);
    const uint32_t n_out = hv[DV_ROWS], n_ids = hv[DV_IDS];
    if (n_out == 0) { finish(); return; }
    c->o_cell_d.ensure((size_t)n_out * 4); c->o_count_d.ensure((size_t)n_out * 4); c->o_n_d.ensure((size_t)(n_out + 1) * 4);
    c->o_off_d.ensure((size_t)(n_out + 1) * 4); c->o_ids_d.ensure((size_t)n_ids * 4 + 16);
    if (!c->defer_fetch) host_rows(n_out, n_ids);
    emit_counts_kernel<<<nblk(n_out + 1, 128), 128, 0, c->s_compute>>>(n_out, c->gstart2.as<uint32_t>(), dv, c->permA.as<uint32_t>(),
                                                                        uo.cell, uo.n, c->o_cell_d.as<uint32_t>(),
                                                                        c->o_count_d.as<uint32_t>(), c->o_n_d.as<uint32_t>());
    const bool defer = c->defer_fetch != 0;       // the table stays on the device until nb200_fetch_counts (nb200_set_defer_fetch)
    if (!defer) {
        CK(cudaMemcpyAsync(c->h_cell.p, c->o_cell_d.p, (size_t)n_out * 4, cudaMemcpyDeviceToHost, c->s_compute));
        CK(cudaMemcpyAsync(c->h_count.p, c->o_count_d.p, (size_t)n_out * 4, cudaMemcpyDeviceToHost, c->s_compute));
    }
    excl_scan_u32(c, c->o_n_d.as<uint32_t>(), c->o_off_d.as<uint32_t>(), n_out + 1);
    if (!defer) CK(cudaMemcpyAsync(c->h_off.p, c->o_off_d.p, (size_t)(n_out + 1) * 4, cudaMemcpyDeviceToHost, c->s_compute));
    emit_ids_kernel<<<nblk(n_out, 128), 128, 0, c->s_compute>>>(n_out, c->gstart2.as<uint32_t>(), c->permA.as<uint32_t>(), lists,
                                                                 c->o_off_d.as<uint32_t>(), c->o_ids_d.as<uint32_t>());
    c->launches += 4;
    if (defer) {
        CK(cudaStreamSynchronize(c->s_compute));
        counts->n_rows = n_out;
        c->dev_rows = n_out; c->dev_ids = n_ids;
        c->fetch_pending = true;
        return;                                   // host pointers of `counts` stay null: nb200_fetch_counts fills them
    }
    CK(cudaMemcpyAsync(c->h_ids.p, c->o_ids_d.p, (size_t)n_ids * 4, cudaMemcpyDeviceToHost, c->s_compute));
    CK(cudaStreamSynchronize(c->s_compute));
    if (c->h_off.p[n_out] != n_ids) throw std::runtime_error("internal: id count of the table disagrees with its offsets");
    c->timing.d2h_bytes += (uint64_t)n_out * 12 + 4 + (uint64_t)n_ids * 4;
    counts->n_rows = n_out;
    c->dev_rows = n_out; c->dev_ids = n_ids;
    finish();
}

static void ensure_read_buffers(nb200_ctx *c, const nb200_reads *r1, const nb200_reads *r2, bool has_key) {
    c->n_reads = r1->n;
    c->paired = r2 != nullptr;
    c->has_key = has_key;
    const uint32_t s1 = is_compact(r1) ? full_stride(r1->words) : r1->stride;      // records are always full on the device
    c->d_r1.ensure(r1->n * (size_t)s1 + 64); c->d_r1len.ensure(r1->n * 2 + 16);
    c->r1 = ReadsDev{c->d_r1.as<uint8_t>(), c->d_r1len.as<uint16_t>(), s1, r1->words};
    if (r2) {
        const uint32_t s2 = is_compact(r2) ? full_stride(r2->words) : r2->stride;
        c->d_r2.ensure(r2->n * (size_t)s2 + 64); c->d_r2len.ensure(r2->n * 2 + 16);
        c->r2 = ReadsDev{c->d_r2.as<uint8_t>(), c->d_r2len.as<uint16_t>(), s2, r2->words};
    } else c->r2 = c->r1;
    if (has_key) c->d_key.ensure(r1->n * 8 + 16);
}

static void validate_reads(const nb200_reads *r, const char *what) {
    if (!r->packed || !r->len) throw std::runtime_error(std::string(what) + ": null buffers");
    if (r->words == 0) throw std::runtime_error(std::string(what) + ": bad layout");
    if (r->stride == 8 * r->words) {                       // compact wire form: side table of the reads with N
        if (r->n_with_n && (!r->n_idx || !r->n_mask)) throw std::runtime_error(std::string(what) + ": compact reads without their N table");
        if (r->n_with_n > r->n || r->n > 0xFFFFFFFFull) throw std::runtime_error(std::string(what) + ": bad N table");
    } else if (r->stride < 12 * r->words || (r->stride & 15)) throw std::runtime_error(std::string(what) + ": bad layout");
    if (r->words * 32 > NB200_MAX_READ_LEN + 31) throw std::runtime_error(std::string(what) + ": reads longer than 500 bases");
}

struct HostInput { const nb200_reads *r1, *r2; const uint64_t *key; };

// Device state of one batch of up to nbmax reads with n_ro mate-orientations, and the wide-read scratch of library L.
// The Smith-Waterman work list starts at 8 items a read (NB200_ITEMS_CAP overrides it: tests force the overflow-and-retry
// path with it) and only grows after an overflow (grown_items_cap).
static void size_batch(nb200_ctx *c, nb200_ctx::BatchBuf &b, uint64_t nbmax, int n_ro, const DevLibrary &L) {
    if (c->items_cap == 0) {
        c->items_cap = (uint32_t)std::max<uint64_t>(1u << 20, std::min<uint64_t>(nbmax * 8, 1ull << 28));
        if (const char *e = getenv("NB200_ITEMS_CAP")) c->items_cap = (uint32_t)std::max(2l, atol(e));
    }
    b.ro.ensure(nbmax * n_ro * sizeof(RoRec));
    b.roB.ensure(nbmax * n_ro * (size_t)2 * kCap * 4);
    b.deferred.ensure(nbmax * 4);
    b.wide_list.ensure(nbmax * 4);
    b.warp_list.ensure(nbmax * 4);
    b.sums.ensure(nbmax * n_ro * sizeof(OriSum));
    b.slow_list.ensure(nbmax * 4);
    b.setup_list.ensure(nbmax * 4);
    b.items.ensure((size_t)c->items_cap * sizeof(SwItem));
    b.sw_pairs.ensure(((size_t)c->items_cap + 64) * 4);      // distinct-window work list
    b.sw_rep.ensure(((size_t)c->items_cap + 64) * 4);        // representative of every candidate
    const size_t warps = (size_t)kWideBlocks * 4;
    c->wide_scratch.ensure(warps * 16 * (size_t)L.dev.n_words * 4);
    c->wide_v.ensure(warps * ((size_t)L.dev.n_words * 32 + 32) * 4);
}

// the work list after an overflow: the measured demand of the batch and some room
static uint32_t grown_items_cap(unsigned long long need) {
    return (uint32_t)std::min<unsigned long long>(need + need / 4 + 1024, 0xFFFFFFF0ull);
}

// The whole hot path for one library.  `in` == nullptr: reads already resident.
static void run_align(nb200_ctx *c, DevLibrary &L, const HostInput *in, double threshold, int disable,
                      nb200_counts *counts) {
    if (!L.host.has_index) throw std::runtime_error("library has no k-mer index (feature dictionary only)");
    const uint64_t n = c->n_reads;
    if (n == 0) {
        c->timing = nb200_timing{};
        aggregate(c, L, 0, nullptr, Rows{}, nullptr, 0, threshold, disable, counts);
        return;
    }
    const int n_mates = c->paired ? 2 : 1, n_ro = n_mates * 2;
    const nb200_config &cfg = L.host.cfg;
    const CallParams cp = call_params(c, L);
    const uint32_t mh = (uint32_t)cfg.max_hits_to_report;
    c->results.ensure(n * sizeof(nb200_read_result) + 64);
    c->feats.ensure(n * (size_t)mh * 4 + 64);
    c->row_nf.ensure(n * 2 + 64);
    c->feats_stride = (int32_t)mh;
    const uint64_t B = c->paired ? (1ull << 20) : (1ull << 21);
    const uint64_t nbmax = std::min<uint64_t>(B, std::max<uint64_t>(n, 1));
    if (in) {   // compact wire form: staging sized once for the largest batch (a reallocation inside the loop would sync)
        if (is_compact(in->r1)) c->stage1.ensure(nbmax * (size_t)in->r1->stride + 64);
        if (in->r2 && is_compact(in->r2)) c->stage2.ensure(nbmax * (size_t)in->r2->stride + 64);
    }
    pin_index_in_l2(c, L);
    for (int attempt = 0; attempt < 3; attempt++) {
        for (auto &b : c->bb) {
            size_batch(c, b, nbmax, n_ro, L);
            b.busy = false;
        }
        CK(cudaMemsetAsync(c->bb[1].ctr, 0, sizeof(Counters), c->s_compute));
        c->timing = nb200_timing{};
        c->launches = 0;
        CK(cudaMemsetAsync(c->d_ctr.p, 0, sizeof(Counters), c->s_compute));
        cudaEvent_t e0 = new_event(c), e1 = new_event(c), e_h2d = new_event(c);
        std::vector<cudaEvent_t> ev, ev_pk;
        if (in) {
            CK(cudaStreamSynchronize(c->s_compute));
            CK(cudaEventRecord(e0, c->s_copy[0]));
            CK(cudaStreamWaitEvent(c->s_copy[1], e0, 0));
        } else {
            CK(cudaEventRecord(e0, c->s_compute));
        }
        size_t nbatch = 0;
        // host input: ramp the batch size up (B/8, B/2, B, B, ...) so the first kernel starts after a small
        // H2D slice instead of waiting for a full batch
        uint64_t nb = 0;
        std::vector<uint64_t> ramp;              // NB200_RAMP="8,3,..." overrides the divisors of the first batches (experiments)
        if (const char *e = getenv("NB200_RAMP")) { for (const char *p = e; *p;) { char *q; const long v = strtol(p, &q, 10); if (q == p) break; ramp.push_back((uint64_t)std::max(1l, v)); p = *q ? q + 1 : q; } }
        for (uint64_t r0 = 0; r0 < n; r0 += nb) {
            uint64_t want = !in ? B : (nbatch == 0 ? B / 8 : (nbatch == 1 ? B / 2 : B));
            if (in && nbatch < ramp.size()) want = std::max<uint64_t>(1024, B / ramp[nbatch]);
            nb = std::min<uint64_t>(want, n - r0);
            if (in) {   // stream this batch's slices ahead of the kernels
                // one copy stream, in order: the link is shared anyway, and with two streams the DMA engines
                // interleave so that batch k+1 delays batch k (measured: second batch ready after 6 ms instead of 1.4)
                cudaStream_t cs = c->s_copy[0];
                c->timing.h2d_bytes += h2d_reads(c, cs, in->r1, c->stage1, c->d_r1.as<uint8_t>(), c->d_r1len.as<uint16_t>(), r0, nb);
                if (in->r2)
                    c->timing.h2d_bytes += h2d_reads(c, cs, in->r2, c->stage2, c->d_r2.as<uint8_t>(), c->d_r2len.as<uint16_t>(), r0, nb);
                if (in->key) {
                    CK(cudaMemcpyAsync(c->d_key.as<uint64_t>() + r0, in->key + r0, nb * 8, cudaMemcpyHostToDevice, cs));
                    c->timing.h2d_bytes += nb * 8;
                }
                cudaEvent_t ec = new_event(c);
                CK(cudaEventRecord(ec, cs));
                CK(cudaStreamWaitEvent(c->s_compute, ec, 0));
                if (r0 + nb >= n) CK(cudaEventRecord(e_h2d, cs));
            }
            cudaEvent_t a = new_event(c), b = new_event(c), t0 = new_event(c), d = new_event(c), e = new_event(c), pk = new_event(c);
            const BatchIO io{c->r1, c->r2, c->results.as<nb200_read_result>() + r0, c->feats.as<int32_t>() + r0 * cp.max_hits,
                             c->row_nf.as<uint16_t>() + r0};
            launch_batch(c, L, cp, io, r0, nb, n_mates, (int)(nbatch & 1), a, b, t0, d, e, pk);
            ev.push_back(a); ev.push_back(b); ev.push_back(t0); ev.push_back(d); ev.push_back(e); ev_pk.push_back(pk);
            nbatch++;
        }
        // every batch's tail done, odd-batch counters folded into the main ones
        for (auto &bbuf : c->bb) if (bbuf.busy && c->overlap) CK(cudaStreamWaitEvent(c->s_compute, bbuf.tail_done, 0));
        merge_counters_kernel<<<1, kCtrSpread, 0, c->s_compute>>>(c->d_ctr.as<Counters>(), c->bb[1].ctr);
        cudaEvent_t e_agg = new_event(c);
        CK(cudaEventRecord(e_agg, c->s_compute));
        // counters (overflow check + max_nf) before the aggregation sizes its sorts
        struct { Counters c; } hc;
        CK(cudaMemcpyAsync(&hc, c->d_ctr.p, sizeof(hc), cudaMemcpyDeviceToHost, c->s_compute));
        CK(cudaStreamSynchronize(c->s_compute));
        c->timing.d2h_bytes += sizeof(hc);
        if (hc.c.overflow) {   // SW work list did not fit: grow to the measured demand and redo
            c->items_cap = grown_items_cap(hc.c.items_max);
            continue;
        }
        aggregate(c, L, n, c->has_key ? c->d_key.as<uint64_t>() : nullptr, Rows{c->feats.as<int32_t>(), nullptr, nullptr, c->row_nf.as<uint16_t>(), mh},
                  nullptr, 0, threshold, disable, counts);
        CK(cudaEventRecord(e1, c->s_compute));
        CK(cudaStreamSynchronize(c->s_compute));
        Counters h2;
        CK(cudaMemcpy(&h2, c->d_ctr.p, sizeof(h2), cudaMemcpyDeviceToHost));
        counts->dropped_empty = h2.dropped_empty;
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, e0, e1)); c->timing.total_ms = ms;
        CK(cudaEventElapsedTime(&ms, e_agg, e1)); c->timing.agg_ms = ms;
        if (in && n) { CK(cudaEventElapsedTime(&ms, e0, e_h2d)); c->timing.h2d_ms = ms; }
        if (getenv("NB200_TRACE")) {   // per-batch timeline relative to the start of the call
            float t_agg = 0;
            CK(cudaEventElapsedTime(&t_agg, e0, e_agg));
            for (size_t i = 0; i + 4 < ev.size(); i += 5) {
                float ta, tb, tt, td, te;
                CK(cudaEventElapsedTime(&ta, e0, ev[i])); CK(cudaEventElapsedTime(&tb, e0, ev[i + 1]));
                CK(cudaEventElapsedTime(&tt, e0, ev[i + 2])); CK(cudaEventElapsedTime(&td, e0, ev[i + 3]));
                CK(cudaEventElapsedTime(&te, e0, ev[i + 4]));
                fprintf(stderr, "[nb200 trace] batch %zu: probe %.2f-%.2f  tail start %.2f sw-end %.2f call-end %.2f ms\n", i / 5, ta, tb, tt, td, te);
            }
            fprintf(stderr, "[nb200 trace] agg start %.2f end %.2f ms\n", t_agg, c->timing.total_ms);
        }
        // stage times are elapsed times on their own streams: with overlap on they add up to more than total_ms
        for (size_t i = 0; i + 4 < ev.size(); i += 5) {
            CK(cudaEventElapsedTime(&ms, ev[i], ev[i + 1])); c->timing.probe_ms += ms;
            CK(cudaEventElapsedTime(&ms, ev[i], ev_pk[i / 5])); c->timing.probe_kernel_ms += ms;
            CK(cudaEventElapsedTime(&ms, ev[i + 2], ev[i + 3])); c->timing.sw_ms += ms;
            CK(cudaEventElapsedTime(&ms, ev[i + 3], ev[i + 4])); c->timing.call_ms += ms;
        }
        for (int i = 0; i < kCtrSpread; i++) { c->timing.probes += h2.probes[i]; c->timing.probe_slots += h2.probe_slots[i]; }
        c->timing.sw_pairs = h2.sw_pairs; c->timing.sw_cells = h2.sw_cells; c->timing.sw_items = h2.sw_pairs + h2.sw_dups;
        c->timing.probe_warp_reads = h2.probe_warp_total;
        c->timing.launches = c->launches;
        c->ev_pool.clear();
        return;
    }
    throw std::runtime_error("Smith-Waterman work list kept overflowing");
}


// ---------------------------------------------------------------------------------------------
// Streaming file path (slab_api.hpp): two slabs in flight per context
// ---------------------------------------------------------------------------------------------
static DevLibrary &lane_lib(nb200_ctx *c, int32_t id) {
    if (id < 0 || id >= (int32_t)c->libs.size()) throw std::runtime_error("bad library id");
    return *c->libs[id];
}
void lane_bind_thread(nb200_ctx *c) { CK(cudaSetDevice(c->device)); }
int lane_max_hits(nb200_ctx *c, int32_t lib_id) { return lane_lib(c, lib_id).host.cfg.max_hits_to_report; }
uint32_t lane_n_features(nb200_ctx *c, int32_t lib_id) { return lane_lib(c, lib_id).host.n_features; }
int lane_host_threads(nb200_ctx *c) { return c->host_threads; }
bool lane_pin(void *p, size_t bytes) {
    if (cudaHostRegister(p, bytes, cudaHostRegisterPortable) == cudaSuccess) return true;
    cudaGetLastError();
    return false;
}
void lane_unpin(void *p) { if (cudaHostUnregister(p) != cudaSuccess) cudaGetLastError(); }
const char *lane_feature_name(nb200_ctx *c, int32_t lib_id, uint32_t fid, uint32_t *len) {
    const std::string &s = lane_lib(c, lib_id).host.feature_names[fid];
    if (len) *len = (uint32_t)s.size();
    return s.data();
}

bool lane_trim(nb200_ctx *c, int32_t lib_id, int *target, double *strictness) {
    const HostLibrary &h = lane_lib(c, lib_id).host;
    if (target) *target = h.trim_target;
    if (strictness) *strictness = h.trim_strictness;
    return h.trim_on;
}

// Grow three arrays that work queued on stream s may still read or write: each gets a new buffer of `bytes`, its first
// `keep` bytes copied over on s; the old buffer goes to `retired`, which the caller frees only when the store is reset.
struct Regrow { DevBuf &buf; size_t bytes, keep; };
static void grow_keep_retire(const Regrow (&a)[3], cudaStream_t s, std::vector<DevBuf> &retired) {
    DevBuf fresh[3];
    for (int i = 0; i < 3; i++) fresh[i].ensure(a[i].bytes);
    for (int i = 0; i < 3; i++) {
        if (a[i].keep) CK(cudaMemcpyAsync(fresh[i].p, a[i].buf.p, a[i].keep, cudaMemcpyDeviceToDevice, s));
        if (a[i].buf.p) retired.push_back(std::move(a[i].buf));
        a[i].buf = std::move(fresh[i]);
    }
}

// Counts mode: append the slab's rows of store li behind its calling kernels, on s_copy[1] (the stream every lane's
// result copies use, so that the appends of the two lanes follow one another).  The store grows geometrically; what it
// must hold is known on the host without a synchronise: its end as of the last segment seen (lane_wait) plus, at most,
// the reads of the other lane's slab in flight and of this one.
static void append_rows(nb200_ctx *c, nb200_ctx::FileLane &F, int li, uint64_t n, const nb200_read_result *res, const int32_t *feats, uint32_t mh) {
    cudaStream_t sd = c->s_copy[1];
    nb200_ctx::RowStore &S = c->rs[(size_t)li];
    uint64_t other = 0;
    for (auto &G : c->lane) if (&G != &F && G.busy && G.hkey) other += G.n_rows_max;
    const uint64_t live_r = S.hi_rows + other, live_i = S.hi_ids + other * S.mh;
    const uint64_t need_r = live_r + n, need_i = live_i + n * mh;
    if (need_r > S.cap_rows || need_i > S.cap_ids) {
        const uint64_t cr = std::max(need_r, 2 * S.cap_rows), ci = std::max(need_i, 2 * S.cap_ids);
        const uint64_t keep_r = std::min(live_r, S.cap_rows), keep_i = std::min(live_i, S.cap_ids);
        grow_keep_retire({{S.key, cr * 8, keep_r * 8}, {S.nf, cr * 4, keep_r * 4}, {S.ids, ci * 4, keep_i * 4}}, sd, S.old);
        S.cap_rows = cr; S.cap_ids = ci;
    }
    c->rs_val.ensure((n + 1) * 8); c->rs_pos.ensure((n + 1) * 8);
    unsigned long long *seg = F.seg.as<unsigned long long>() + 5 * (size_t)li;
    CK(cudaMemsetAsync(seg, 0, 5 * 8, sd));
    row_flag_kernel<<<nblk(n + 1, 256), 256, 0, sd>>>((uint32_t)n, F.key.as<uint64_t>(), res, feats, mh, S.na.as<uint8_t>(),
                                                      c->rs_val.as<uint64_t>(), seg + 4);
    size_t bytes = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, bytes, c->rs_val.as<uint64_t>(), c->rs_pos.as<uint64_t>(), (int)(n + 1), sd));
    c->rs_tmp.ensure(bytes);
    CK(cub::DeviceScan::ExclusiveSum(c->rs_tmp.p, bytes, c->rs_val.as<uint64_t>(), c->rs_pos.as<uint64_t>(), (int)(n + 1), sd));
    if (n) row_scatter_kernel<<<nblk(n, 256), 256, 0, sd>>>((uint32_t)n, F.key.as<uint64_t>(), feats, mh, c->rs_pos.as<uint64_t>(),
                                                     S.hdr.as<unsigned long long>(), S.key.as<uint64_t>(), S.nf.as<uint32_t>(), S.ids.as<int32_t>());
    row_advance_kernel<<<1, 1, 0, sd>>>(c->rs_pos.as<uint64_t>() + n, S.hdr.as<unsigned long long>(), seg);
    CK(cudaMemcpyAsync(F.h_seg.p + 5 * (size_t)li, seg, 5 * 8, cudaMemcpyDeviceToHost, sd));
    c->launches += 4;
}

// ---- cell-barcode correction shared by the whole-batch path (cb_run) and the slabs of fastq-to-counts ---------------
struct MaxU32 {
    __host__ __device__ __forceinline__ uint32_t operator()(uint32_t a, uint32_t b) const { return a > b ? a : b; }
};

// Phases 1 and 2 (barcode.cuh) over n barcodes on stream s: counters and multi-candidate flags are zeroed first; the
// miss count stays on the device.  inval may be null (inval_cap 0), hit and elig too.
static void cb_launch(nb200_ctx *c, const WlDev &W, cudaStream_t s, const uint8_t *chars, const uint8_t *qual, const uint8_t *elig,
                      uint64_t n, uint64_t *keys, int32_t *idx, uint8_t *status, uint32_t *miss, uint32_t *inval, uint32_t inval_cap,
                      uint8_t *hit, uint8_t *multi, CbCounters *ctr) {
    CK(cudaMemsetAsync(ctr, 0, sizeof(CbCounters), s));
    CK(cudaMemsetAsync(multi, 0, n + 16, s));
    if (!n) return;
    cb_exact_kernel<<<nblk(n, 256), 256, 0, s>>>(W, chars, elig, n, keys, idx, status, miss, inval, inval_cap, hit, ctr);
    cb_hamming_kernel<<<c->sm_count * 8, 128, 0, s>>>(W, qual, keys, miss, idx, status, multi, ctr);
    CK(cudaGetLastError());
    c->launches += 2;
}

// Phase 3, the reference's correction_cache: list = m reads with several candidates in file order (indices into keys /
// out_idx); afterwards each of them carries the choice of the first one with its raw barcode.  On s_compute.
static void cb_first_decides(nb200_ctx *c, const uint32_t *list, const uint64_t *keys, uint32_t m, int32_t *out_idx) {
    cudaStream_t s = c->s_compute;
    c->k64A.ensure((size_t)m * 8 + 16); c->k64B.ensure((size_t)m * 8 + 16);
    c->k32A.ensure((size_t)m * 4 + 16); c->k32B.ensure((size_t)m * 4 + 16); c->head.ensure((size_t)m * 4 + 16);
    cb_gather_keys_kernel<<<nblk(m, 256), 256, 0, s>>>(list, keys, m, c->k64A.as<uint64_t>());
    cub_sort64(c, c->k64A.as<uint64_t>(), c->k64B.as<uint64_t>(), list, c->k32A.as<uint32_t>(), m, 64);   // stable
    cb_run_heads_kernel<<<nblk(m, 256), 256, 0, s>>>(c->k64B.as<uint64_t>(), m, c->k32B.as<uint32_t>());
    size_t bytes = 0;
    CK(cub::DeviceScan::InclusiveScan(nullptr, bytes, c->k32B.as<uint32_t>(), c->head.as<uint32_t>(), MaxU32(), (int)m, s));
    c->cub_tmp.ensure(bytes);
    CK(cub::DeviceScan::InclusiveScan(c->cub_tmp.p, bytes, c->k32B.as<uint32_t>(), c->head.as<uint32_t>(), MaxU32(), (int)m, s));
    cb_propagate_kernel<<<nblk(m, 256), 256, 0, s>>>(c->k32A.as<uint32_t>(), c->head.as<uint32_t>(), m, out_idx);
    CK(cudaGetLastError());
    c->launches += 8;
}

// fastq-to-counts, per slab (inside lane_submit, on s_compute behind the slab's uploads): correct the barcodes, turn the
// host's UMI keys into cell << 32 | umi, log the reads with several candidates.  No host synchronise: the log's capacity
// is bounded on the host (its end as of the last slab seen plus the reads of the slabs in flight).
static void lane_cb_slab(nb200_ctx *c, nb200_ctx::FileLane &F, uint64_t n) {
    cudaStream_t s = c->s_compute;
    uint64_t other = 0;
    for (auto &G : c->lane) if (&G != &F && G.busy && G.hcb) other += G.n_rows_max;
    const uint64_t need = c->tx_hi + other + n;
    if (need > c->tx_cap) {                          // grow: copy on s_compute (every log write is on it), free at the end
        const uint64_t cap = std::max(need, 2 * c->tx_cap);
        const uint64_t keep = std::min(c->tx_hi + other, c->tx_cap);
        grow_keep_retire({{c->tx_key, cap * 8, keep * 8}, {c->tx_ord, cap * 8, keep * 8}, {c->tx_choice, cap * 4, keep * 4}}, s, c->tx_old);
        c->tx_cap = cap;
    }
    const uint64_t nb = std::max<uint64_t>(n, 1);
    F.cb_raw.ensure(nb * 8); F.cb_idx.ensure(nb * 4); F.cb_st.ensure(nb); F.cb_miss.ensure(nb * 4); F.cb_multi.ensure(nb + 16);
    F.cb_ctr.ensure(sizeof(CbCounters));
    CbCounters *ctr = F.cb_ctr.as<CbCounters>();
    cb_launch(c, c->tx_wl, s, F.cb.as<uint8_t>(), F.cbq.as<uint8_t>(), nullptr, n, F.cb_raw.as<uint64_t>(), F.cb_idx.as<int32_t>(),
              F.cb_st.as<uint8_t>(), F.cb_miss.as<uint32_t>(), nullptr, 0, nullptr, F.cb_multi.as<uint8_t>(), ctr);
    if (n) {
        cb_key_kernel<<<nblk(n, 256), 256, 0, s>>>((uint32_t)n, F.cb_st.as<uint8_t>(), F.cb_idx.as<int32_t>(), F.cb_multi.as<uint8_t>(),
                                                   F.cb_raw.as<uint64_t>(), F.seq << 21, F.key.as<uint64_t>(), c->tx_n.as<unsigned long long>(),
                                                   c->tx_key.as<uint64_t>(), c->tx_ord.as<uint64_t>(), c->tx_choice.as<int32_t>(), ctr);
        CK(cudaGetLastError());
        c->launches++;
    }
    // (read after lane_wait: the lane's done event follows these copies through s_compute's tail)
    CK(cudaMemcpyAsync(F.h_cb.p, ctr, sizeof(CbCounters), cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(F.h_cb.p + 8, c->tx_n.p, 8, cudaMemcpyDeviceToHost, s));
}

void lane_submit(nb200_ctx *c, int lane, const nb200_reads *r1, const nb200_reads *r2, const int32_t *lib_ids, int n_libs,
                 nb200_read_result *const *out_res, int32_t *const *out_feats, uint16_t *const *len1, uint16_t *const *len2,
                 const uint64_t *key, const uint8_t *cb, const uint8_t *cb_qual, uint64_t seq) {
    nb200_ctx::FileLane &F = c->lane[lane];
    if (F.busy) throw std::runtime_error("lane is busy");
    if (key && c->rs.size() < (size_t)n_libs) throw std::runtime_error("counts mode without lane_rows_begin");
    if (cb && (!key || !cb_qual || !c->tx_table.p)) throw std::runtime_error("barcodes without lane_cb_begin");
    validate_reads(r1, "r1");
    if (r2) { validate_reads(r2, "r2"); if (r2->n != r1->n) throw std::runtime_error("r1 and r2 differ in read count"); }
    const uint64_t n = r1->n;
    if (is_compact(r1) || (r2 && is_compact(r2))) throw std::runtime_error("file lanes take full records");
    if (n > (1ull << 21) || (r2 && n > (1ull << 20))) throw std::runtime_error("slab larger than a batch");
    if (!F.h2d_done) { CK(cudaEventCreateWithFlags(&F.h2d_done.h, cudaEventDisableTiming)); CK(cudaEventCreateWithFlags(&F.done.h, cudaEventDisableTiming)); }
    F.h_ctr.ensure((size_t)n_libs);
    F.hr1 = *r1; F.paired = r2 != nullptr; if (r2) F.hr2 = *r2;
    F.libs.assign(lib_ids, lib_ids + n_libs);
    F.out_res.clear(); F.out_feats.clear();
    if (out_res) F.out_res.assign(out_res, out_res + n_libs);
    if (out_feats) F.out_feats.assign(out_feats, out_feats + n_libs);
    F.hkey = key; F.n_rows_max = key ? n : 0;
    F.hcb = cb; F.hcbq = cb_qual; F.seq = seq;
    if (cb) F.h_cb.ensure(9);
    if (key) F.h_seg.ensure(5 * (size_t)n_libs);
    F.hlen1.clear(); F.hlen2.clear();
    if (len1) F.hlen1.assign(len1, len1 + n_libs);
    if (len2 && r2) F.hlen2.assign(len2, len2 + n_libs);
    F.res.resize(std::max<size_t>(F.res.size(), (size_t)n_libs)); F.feats.resize(F.res.size()); F.nf.resize(F.res.size());
    const int n_mates = r2 ? 2 : 1, n_ro = n_mates * 2;
    // reads up, once for all libraries
    cudaStream_t sh = c->s_copy[0], sd = c->s_copy[1];
    F.r1.ensure(n * (size_t)r1->stride + 64); F.l1.ensure(n * 2 + 16);
    if (n) {
        CK(cudaMemcpyAsync(F.r1.p, r1->packed, n * (size_t)r1->stride, cudaMemcpyHostToDevice, sh));
        CK(cudaMemcpyAsync(F.l1.p, r1->len, n * 2, cudaMemcpyHostToDevice, sh));
    }
    BatchIO io{};
    io.r1 = ReadsDev{F.r1.as<uint8_t>(), F.l1.as<uint16_t>(), r1->stride, r1->words};
    io.r2 = io.r1;
    if (r2) {
        F.r2.ensure(n * (size_t)r2->stride + 64); F.l2.ensure(n * 2 + 16);
        if (n) {
            CK(cudaMemcpyAsync(F.r2.p, r2->packed, n * (size_t)r2->stride, cudaMemcpyHostToDevice, sh));
            CK(cudaMemcpyAsync(F.l2.p, r2->len, n * 2, cudaMemcpyHostToDevice, sh));
        }
        io.r2 = ReadsDev{F.r2.as<uint8_t>(), F.l2.as<uint16_t>(), r2->stride, r2->words};
    }
    if (key) {
        F.key.ensure(n * 8 + 16); F.seg.ensure(5 * 8 * (size_t)n_libs);
        if (n) CK(cudaMemcpyAsync(F.key.p, key, n * 8, cudaMemcpyHostToDevice, sh));
    }
    if (cb) {
        const size_t L = (size_t)c->tx_wl.cb_len;
        F.cb.ensure(n * L + 16); F.cbq.ensure(n * L + 16);
        if (n) {
            CK(cudaMemcpyAsync(F.cb.p, cb, n * L, cudaMemcpyHostToDevice, sh));
            CK(cudaMemcpyAsync(F.cbq.p, cb_qual, n * L, cudaMemcpyHostToDevice, sh));
        }
    }
    if (len1 && n) {      // per-library lengths: all up before the first kernel
        F.l1v.resize(std::max<size_t>(F.l1v.size(), (size_t)n_libs)); F.l2v.resize(F.l1v.size());
        for (int li = 0; li < n_libs; li++) {
            F.l1v[li].ensure(n * 2 + 16);
            CK(cudaMemcpyAsync(F.l1v[li].p, len1[li], n * 2, cudaMemcpyHostToDevice, sh));
            if (r2 && len2) { F.l2v[li].ensure(n * 2 + 16); CK(cudaMemcpyAsync(F.l2v[li].p, len2[li], n * 2, cudaMemcpyHostToDevice, sh)); }
        }
    }
    CK(cudaEventRecord(F.h2d_done, sh));
    CK(cudaStreamWaitEvent(c->s_compute, F.h2d_done, 0));
    if (cb) lane_cb_slab(c, F, n);                  // the keys are final before any library's rows are appended
    nb200_ctx::BatchBuf &B = c->bb[lane];
    const uint64_t nbmax = std::max<uint64_t>(n, 1);
    for (int li = 0; li < n_libs; li++) {
        DevLibrary &L = lane_lib(c, lib_ids[li]);
        if (!L.host.has_index) throw std::runtime_error("library has no k-mer index (feature dictionary only)");
        const CallParams cp = call_params(c, L);
        const uint32_t mh = (uint32_t)cp.max_hits;
        F.res[li].ensure(nbmax * sizeof(nb200_read_result) + 64);
        F.feats[li].ensure(nbmax * (size_t)mh * 4 + 64);
        F.nf[li].ensure(nbmax * 2 + 64);
        size_batch(c, B, nbmax, n_ro, L);
        pin_index_in_l2(c, L);
        if (B.busy && c->overlap) CK(cudaStreamWaitEvent(c->s_compute, B.tail_done, 0));
        CK(cudaMemsetAsync(B.ctr, 0, sizeof(Counters), c->s_compute));
        io.res = F.res[li].as<nb200_read_result>(); io.feats = F.feats[li].as<int32_t>(); io.nf = F.nf[li].as<uint16_t>();
        if (len1 && n) {
            io.r1.len = F.l1v[li].as<uint16_t>();
            if (r2) io.r2.len = len2 ? F.l2v[li].as<uint16_t>() : F.l2.as<uint16_t>(); else io.r2 = io.r1;
        }
        if (n) launch_batch(c, L, cp, io, 0, n, n_mates, lane, nullptr, nullptr, nullptr, nullptr, nullptr);
        else { CK(cudaEventRecord(B.tail_done, c->s_compute)); B.busy = true; }
        // results down, behind the tail of this library's kernels
        CK(cudaStreamWaitEvent(sd, B.tail_done, 0));
        if (n) {
            if (out_res && out_res[li]) CK(cudaMemcpyAsync(out_res[li], io.res, n * sizeof(nb200_read_result), cudaMemcpyDeviceToHost, sd));
            if (out_feats && out_feats[li]) CK(cudaMemcpyAsync(out_feats[li], io.feats, n * (size_t)mh * 4, cudaMemcpyDeviceToHost, sd));
        }
        if (key) append_rows(c, F, li, n, io.res, io.feats, mh);
        CK(cudaMemcpyAsync(&F.h_ctr.p[li], B.ctr, sizeof(Counters), cudaMemcpyDeviceToHost, sd));
        // the next library (or the next slab on this lane) resets B.ctr: not before this copy has read it
        CK(cudaEventRecord(F.done, sd));
        CK(cudaStreamWaitEvent(c->s_compute, F.done, 0));
    }
    CK(cudaEventRecord(F.done, sd));
    F.busy = true;
}

void lane_wait(nb200_ctx *c, int lane) {
    nb200_ctx::FileLane &F = c->lane[lane];
    if (!F.busy) return;
    for (int attempt = 0;; attempt++) {
        CK(cudaEventSynchronize(F.done));
        F.busy = false;
        if (F.hkey)                                     // counts mode: where the stores end now (a re-run appends anew)
            for (size_t li = 0; li < F.libs.size(); li++) {
                const unsigned long long *s = F.h_seg.p + 5 * li;
                nb200_ctx::RowStore &S = c->rs[li];
                S.hi_rows = std::max<uint64_t>(S.hi_rows, s[0] + s[1]);
                S.hi_ids = std::max<uint64_t>(S.hi_ids, s[2] + s[3]);
            }
        if (F.hcb) {
            c->tx_hi = std::max<uint64_t>(c->tx_hi, F.h_cb.p[8]);
            // a pair fastq-to-bam writes (barcode corrected) that it or align on its BAM refuses: CbCounters::pad
            const unsigned long long bad = F.h_cb.p[7];
            if (bad & kTenxLongName) throw std::runtime_error("read name longer than 254 bytes");
            if (bad & kTenxLongRead) throw std::runtime_error("read longer than 500 bases");
        }
        unsigned long long need = 0;
        for (size_t li = 0; li < F.libs.size(); li++)
            if (F.h_ctr.p[li].overflow) need = std::max(need, F.h_ctr.p[li].items_max);
        if (!need) return;
        if (attempt >= 3) throw std::runtime_error("Smith-Waterman work list kept overflowing");
        // the work list did not fit: grow it to the measured demand (cudaFree waits for the other lane) and redo the slab
        c->items_cap = grown_items_cap(need);
        const nb200_reads r1 = F.hr1, r2 = F.hr2;
        const std::vector<int32_t> libs = F.libs;
        const std::vector<nb200_read_result *> orr = F.out_res;
        const std::vector<int32_t *> of = F.out_feats;
        const std::vector<uint16_t *> h1 = F.hlen1, h2 = F.hlen2;
        lane_submit(c, lane, &r1, F.paired ? &r2 : nullptr, libs.data(), (int)libs.size(), orr.empty() ? nullptr : orr.data(),
                    of.empty() ? nullptr : of.data(), h1.empty() ? nullptr : h1.data(), h2.empty() ? nullptr : h2.data(), F.hkey,
                    F.hcb, F.hcbq, F.seq);
    }
}

void lane_rows_begin(nb200_ctx *c, const int32_t *lib_ids, int n_libs) {
    CK(cudaSetDevice(c->device));
    for (auto &S : c->rs) S.reset();                // (a previous call's stores)
    c->rs.resize((size_t)n_libs);
    for (int li = 0; li < n_libs; li++) {
        const HostLibrary &h = lane_lib(c, lib_ids[li]).host;
        nb200_ctx::RowStore &S = c->rs[(size_t)li];
        S.mh = (uint32_t)std::max(1, h.cfg.max_hits_to_report);
        std::vector<uint8_t> na(h.feature_names.size() + 1, 0);
        for (size_t f = 0; f < h.feature_names.size(); f++) {
            const std::string &nm = h.feature_names[f];
            // a name the per-read TSV cannot carry as one token: `report` would read other names (or other rows)
            if (nm.find_first_of(",\t\n\r") != std::string::npos)
                throw std::runtime_error("feature name \"" + nm + "\" contains a comma, tab or line break: counts need names the per-read TSV can carry");
            na[f] = pandas_na(nm) ? 1 : 0;
        }
        S.na.ensure(na.size());
        CK(cudaMemcpy(S.na.p, na.data(), na.size(), cudaMemcpyHostToDevice));
        S.hdr.ensure(16);
        CK(cudaMemset(S.hdr.p, 0, 16));
    }
    c->rs_val.ensure(((size_t)1 << 17) * 8 + 64); c->rs_pos.ensure(((size_t)1 << 17) * 8 + 64);
    CK(cudaDeviceSynchronize());                    // (flags and store ends in place before the lanes' streams read them)
}

void lane_rows_segments(nb200_ctx *c, int lane, RowSeg *out) {
    const nb200_ctx::FileLane &F = c->lane[lane];
    for (size_t li = 0; li < F.libs.size(); li++) {
        const unsigned long long *s = F.h_seg.p + 5 * li;
        out[li].row0 = s[0]; out[li].rows = s[1]; out[li].id0 = s[2]; out[li].ids = s[3]; out[li].called = s[4];
    }
}

// peer access where the devices allow it (cudaMemcpyPeerAsync stages through the host otherwise); current device = ctxs[0]'s
static void enable_peers(const std::vector<nb200_ctx *> &ctxs) {
    const nb200_ctx *c = ctxs[0];
    for (nb200_ctx *x : ctxs)
        if (x->device != c->device) {
            int can = 0;
            CK(cudaDeviceCanAccessPeer(&can, c->device, x->device));
            if (can) {
                const cudaError_t e = cudaDeviceEnablePeerAccess(x->device, 0);
                if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CK(e);
                cudaGetLastError();
            }
        }
}

void lane_rows_count(const std::vector<nb200_ctx *> &ctxs, int li, int32_t lib_id, const std::vector<RowSeg> &segs,
                     const std::vector<uint32_t> &cell_rank, double threshold, int umi_flags, nb200_counts *counts, uint64_t *rows,
                     bool tenx) {
    nb200_ctx *c = ctxs[0];
    for (nb200_ctx *x : ctxs) { CK(cudaSetDevice(x->device)); CK(cudaStreamSynchronize(x->s_copy[1])); }
    CK(cudaSetDevice(c->device));
    DevLibrary &L = lane_lib(c, lib_id);
    uint64_t R = 0, I = 0;
    for (const RowSeg &s : segs) { R += s.rows; I += s.ids; }
    *rows = R;
    if (R > 0x7FFFFFF0ull) throw LimitError("more than 2^31 rows for one library (CUB item counts are int)");
    if (I > 0xFFFFFFF0ull) throw LimitError("more than 2^32 feature names in the rows of one library");
    c->timing = nb200_timing{};
    c->launches = 0;
    c->gen_key.ensure(R * 8 + 16); c->gen_nf.ensure((R + 1) * 4 + 16); c->gen_off.ensure((R + 1) * 4 + 16); c->gen_feats.ensure(I * 4 + 16);
    enable_peers(ctxs);
    // gather in slab order (= per-read TSV order); runs of segments that lie back to back in one store go as one copy
    cudaStream_t s = c->s_compute;
    uint64_t at_r = 0, at_i = 0;
    std::vector<uint64_t> run_row, run_base;       // fastq-to-counts: where each run's rows start, and its context's log
    for (size_t a = 0; a < segs.size();) {
        size_t b = a + 1;
        while (b < segs.size() && segs[b].ctx == segs[a].ctx && segs[b].row0 == segs[b - 1].row0 + segs[b - 1].rows &&
               segs[b].id0 == segs[b - 1].id0 + segs[b - 1].ids) b++;
        uint64_t nr = 0, ni = 0;
        for (size_t j = a; j < b; j++) { nr += segs[j].rows; ni += segs[j].ids; }
        const nb200_ctx *x = ctxs[(size_t)segs[a].ctx];
        const nb200_ctx::RowStore &S = x->rs[(size_t)li];
        auto copy = [&](void *dst, const void *src, size_t bytes) {
            if (!bytes) return;
            if (x->device == c->device) CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, s));
            else CK(cudaMemcpyPeerAsync(dst, c->device, src, x->device, bytes, s));
        };
        copy(c->gen_key.as<uint64_t>() + at_r, S.key.as<uint64_t>() + segs[a].row0, nr * 8);
        copy(c->gen_nf.as<uint32_t>() + at_r, S.nf.as<uint32_t>() + segs[a].row0, nr * 4);
        copy(c->gen_feats.as<int32_t>() + at_i, S.ids.as<int32_t>() + segs[a].id0, ni * 4);
        if (tenx && nr) { run_row.push_back(at_r); run_base.push_back(c->tx_base.at((size_t)segs[a].ctx)); }
        at_r += nr; at_i += ni;
        a = b;
    }
    CK(cudaMemsetAsync(c->gen_nf.as<uint32_t>() + R, 0, 4, s));
    excl_scan_u32(c, c->gen_nf.as<uint32_t>(), c->gen_off.as<uint32_t>(), (uint32_t)(R + 1));
    DevBuf runs, dropped;
    if (R) {
        c->rs_rank.ensure(cell_rank.size() * 4 + 16);
        CK(cudaMemcpyAsync(c->rs_rank.p, cell_rank.data(), cell_rank.size() * 4, cudaMemcpyHostToDevice, s));
        if (tenx) {
            const uint32_t n_runs = (uint32_t)run_row.size();
            run_row.push_back(R);
            runs.ensure((run_row.size() + run_base.size()) * 8);
            dropped.ensure(8);
            CK(cudaMemcpyAsync(runs.p, run_row.data(), run_row.size() * 8, cudaMemcpyHostToDevice, s));
            CK(cudaMemcpyAsync(runs.as<uint64_t>() + run_row.size(), run_base.data(), run_base.size() * 8, cudaMemcpyHostToDevice, s));
            CK(cudaMemsetAsync(dropped.p, 0, 8, s));
            cb_remap_kernel<<<nblk(R, 256), 256, 0, s>>>(R, c->gen_key.as<uint64_t>(), c->rs_rank.as<uint32_t>(), c->tx_dec.as<int32_t>(),
                                                          runs.as<uint64_t>(), runs.as<uint64_t>() + run_row.size(), n_runs,
                                                          dropped.as<unsigned long long>());
        } else {
            cell_rank_kernel<<<nblk(R, 256), 256, 0, s>>>(R, c->gen_key.as<uint64_t>(), c->rs_rank.as<uint32_t>());
        }
        c->launches++;
    }
    CK(cudaMemsetAsync(c->d_ctr.p, 0, sizeof(Counters), s));
    // the aligner writes nimble_score = 1 for every row: score NULL
    aggregate(c, L, R, c->gen_key.as<uint64_t>(), Rows{c->gen_feats.as<int32_t>(), c->gen_off.as<uint32_t>(), nullptr, nullptr, 0}, nullptr,
              0, threshold, umi_flags, counts);
    CK(cudaStreamSynchronize(s));
    Counters h2;
    CK(cudaMemcpy(&h2, c->d_ctr.p, sizeof(h2), cudaMemcpyDeviceToHost));
    counts->dropped_empty = h2.dropped_empty;
    if (dropped.p) {                                // rows whose cell is a pandas NA token: report never reads them
        unsigned long long d = 0;
        CK(cudaMemcpy(&d, dropped.p, 8, cudaMemcpyDeviceToHost));
        *rows = R - d;
    }
    // the stores of this library are done with
    for (nb200_ctx *x : ctxs) {
        CK(cudaSetDevice(x->device));
        x->rs[(size_t)li].reset();
    }
    CK(cudaSetDevice(c->device));
}

// ---------------------------------------------------------------------------------------------
// fastq-to-bam: whitelist table + barcode correction pipeline (barcode.cuh)
// ---------------------------------------------------------------------------------------------
// key of a whitelist line of length cb_len (3-bit codes: integer order == byte order); throws for a byte outside ACGTN
static uint64_t wl_key(const std::string &e, size_t line) {
    uint64_t key = 0;
    for (char ch : e) {
        const uint32_t code = cb_code((uint8_t)ch);
        if (code == 7u) throw std::runtime_error("whitelist line " + std::to_string(line + 1) + " has a base outside ACGTN: " + e);
        key = (key << 3) | code;
    }
    return key;
}

// the open-addressing table of the lines of length cb_len (first line wins for duplicates, as set() keeps one)
static std::vector<WlSlot> wl_slots(const std::vector<std::string> &entries, int cb_len, uint64_t *n_unique) {
    if (cb_len < 1 || cb_len > kCbMaxLen) throw std::runtime_error("cb_len must be 1..21");
    if (entries.size() >= 0x7FFFFFFFull) throw LimitError("whitelist has 2^31 or more lines");
    uint64_t same = 0;
    for (const auto &e : entries) same += (int)e.size() == cb_len;
    uint64_t slots = 1024;
    while (slots < same * 2 + 2) slots <<= 1;
    std::vector<WlSlot> tab(slots, WlSlot{kCbEmpty, 0, 0});
    const uint64_t mask = slots - 1;
    *n_unique = 0;
    for (size_t i = 0; i < entries.size(); i++) {
        const std::string &e = entries[i];
        if ((int)e.size() != cb_len) continue;                  // can never equal a raw barcode or a variant of one
        const uint64_t key = wl_key(e, i);
        uint64_t s = cb_hash(key) & mask;
        while (tab[s].key != kCbEmpty && tab[s].key != key) s = (s + 1) & mask;
        if (tab[s].key == kCbEmpty) { tab[s].key = key; tab[s].idx = (uint32_t)i; ++*n_unique; }   // set(): first line wins
    }
    return tab;
}

static std::unique_ptr<DevWhitelist> build_whitelist(nb200_ctx *c, std::vector<std::string> &&entries, int cb_len) {
    auto W = std::make_unique<DevWhitelist>();
    const std::vector<WlSlot> tab = wl_slots(entries, cb_len, &W->n_unique);
    W->entries = std::move(entries);
    W->cb_len = cb_len;
    const uint64_t slots = tab.size();
    W->n_slots = slots;
    W->table.ensure(slots * sizeof(WlSlot));
    CK(cudaMemcpyAsync(W->table.p, tab.data(), slots * sizeof(WlSlot), cudaMemcpyHostToDevice, c->s_compute));
    CK(cudaStreamSynchronize(c->s_compute));
    W->dev.table = W->table.as<WlSlot>();
    W->dev.mask = slots - 1;
    W->dev.cb_len = cb_len;
    return W;
}

// ---- fastq-to-counts: the whitelist on every context, the cache rule over every context's log (slab_api.hpp) ----------
// the multi-candidate log back to empty, its buffers, outgrown buffers and decisions freed (current device: c's)
static void reset_cb_log(nb200_ctx *c) {
    for (DevBuf *b : {&c->tx_key, &c->tx_ord, &c->tx_choice, &c->tx_dec}) b->release();
    c->tx_old.clear();
    c->tx_cap = c->tx_hi = 0;
    c->tx_base.clear();
}

void lane_cb_begin(const std::vector<nb200_ctx *> &ctxs, const std::vector<std::string> &whitelist, int cb_len,
                   std::vector<uint32_t> *rank, std::vector<std::string> *cells) {
    uint64_t n_unique = 0;
    const std::vector<WlSlot> tab = wl_slots(whitelist, cb_len, &n_unique);
    for (nb200_ctx *c : ctxs) {
        CK(cudaSetDevice(c->device));
        reset_cb_log(c);
        c->tx_table.ensure(tab.size() * sizeof(WlSlot));
        CK(cudaMemcpy(c->tx_table.p, tab.data(), tab.size() * sizeof(WlSlot), cudaMemcpyHostToDevice));
        c->tx_wl = WlDev{c->tx_table.as<WlSlot>(), tab.size() - 1, cb_len};
        c->tx_n.ensure(8);
        CK(cudaMemset(c->tx_n.p, 0, 8));
    }
    CK(cudaSetDevice(ctxs[0]->device));
    // cells: the distinct lines in byte order (= key order), pandas-NA tokens left out (report drops such a cell)
    std::vector<std::pair<uint64_t, uint32_t>> by_key;
    by_key.reserve(n_unique);
    for (size_t i = 0; i < whitelist.size(); i++)
        if ((int)whitelist[i].size() == cb_len) by_key.emplace_back(wl_key(whitelist[i], i), (uint32_t)i);
    std::sort(by_key.begin(), by_key.end());
    rank->assign(whitelist.size(), 0xFFFFFFFFu);
    cells->clear();
    for (size_t j = 0; j < by_key.size(); j++) {
        const uint32_t i = by_key[j].second;
        if (j && by_key[j].first == by_key[j - 1].first) { (*rank)[i] = (*rank)[by_key[j - 1].second]; continue; }
        if (pandas_na(whitelist[i])) continue;
        (*rank)[i] = (uint32_t)cells->size();
        cells->push_back(whitelist[i]);
    }
}

void lane_cb_counters(nb200_ctx *c, int lane, uint64_t *out6) {
    const unsigned long long *h = c->lane[lane].h_cb.p;               // CbCounters: n_miss n_inval perfect corrected none n_multi probes
    out6[0] = h[2]; out6[1] = h[3]; out6[2] = h[4]; out6[3] = h[0]; out6[4] = h[5]; out6[5] = h[6];
}

__global__ void iota_u32_kernel(uint32_t n, uint32_t *__restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = i;
}

void lane_cb_resolve(const std::vector<nb200_ctx *> &ctxs) {
    nb200_ctx *c = ctxs[0];
    std::vector<uint64_t> cnt(ctxs.size());
    for (size_t d = 0; d < ctxs.size(); d++) {
        CK(cudaSetDevice(ctxs[d]->device));
        CK(cudaStreamSynchronize(ctxs[d]->s_compute));
        CK(cudaMemcpy(&cnt[d], ctxs[d]->tx_n.p, 8, cudaMemcpyDeviceToHost));
    }
    CK(cudaSetDevice(c->device));
    c->tx_base.assign(ctxs.size(), 0);
    uint64_t E = 0;
    for (size_t d = 0; d < ctxs.size(); d++) { c->tx_base[d] = E; E += cnt[d]; }
    if (E > 0x7FFFFFF0ull) throw LimitError("more than 2^31 reads whose cell barcode has several candidates");
    c->tx_dec.ensure(E * 4 + 16);
    if (!E) return;
    // every log on the first context, in context order (entry j of context d is decision tx_base[d] + j)
    DevBuf key, ord, sorted, perm;
    key.ensure(E * 8); ord.ensure(E * 8); sorted.ensure(E * 8); perm.ensure(E * 8);
    enable_peers(ctxs);
    cudaStream_t s = c->s_compute;
    for (size_t d = 0; d < ctxs.size(); d++) {
        const nb200_ctx *x = ctxs[d];
        const uint64_t at = c->tx_base[d], n = cnt[d];
        auto copy = [&](void *dst, const void *src, size_t bytes) {
            if (!bytes) return;
            if (x->device == c->device) CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, s));
            else CK(cudaMemcpyPeerAsync(dst, c->device, src, x->device, bytes, s));
        };
        copy(key.as<uint64_t>() + at, x->tx_key.p, n * 8);
        copy(ord.as<uint64_t>() + at, x->tx_ord.p, n * 8);
        copy(c->tx_dec.as<int32_t>() + at, x->tx_choice.p, n * 4);
    }
    // entries in file order, then the first of each raw barcode decides (a re-run slab's duplicates agree with the original)
    iota_u32_kernel<<<nblk(E, 256), 256, 0, s>>>((uint32_t)E, perm.as<uint32_t>() + E);
    cub_sort64(c, ord.as<uint64_t>(), sorted.as<uint64_t>(), perm.as<uint32_t>() + E, perm.as<uint32_t>(), (uint32_t)E, 64);
    cb_first_decides(c, perm.as<uint32_t>(), key.as<uint64_t>(), (uint32_t)E, c->tx_dec.as<int32_t>());
    CK(cudaStreamSynchronize(s));
}

void lane_cb_end(const std::vector<nb200_ctx *> &ctxs) {
    for (nb200_ctx *c : ctxs) {
        CK(cudaSetDevice(c->device));
        c->tx_table.release();
        reset_cb_log(c);
    }
    CK(cudaSetDevice(ctxs[0]->device));
}

static DevWhitelist &get_wl(const nb200_ctx *c, int32_t id) {
    if (id < 0 || id >= (int32_t)c->wls.size() || !c->wls[id]) throw std::runtime_error("unknown whitelist id");
    return *c->wls[id];
}

static void cb_upload(nb200_ctx *c, int cb_len, const char *cb, const uint8_t *qual, const uint8_t *eligible, uint64_t n,
                      nb200_cb_stats *st) {
    if (n > 0x7FFFFFF0ull) throw LimitError("more than 2^31 reads in one barcode batch (CUB item counts are int)");
    c->cb_chars.ensure(n * (size_t)cb_len + 16);
    c->cb_qual.ensure(n * (size_t)cb_len + 16);
    c->cb_elig.ensure(n + 16);
    if (n) {
        CK(cudaMemcpyAsync(c->cb_chars.p, cb, n * (size_t)cb_len, cudaMemcpyHostToDevice, c->s_compute));
        CK(cudaMemcpyAsync(c->cb_qual.p, qual, n * (size_t)cb_len, cudaMemcpyHostToDevice, c->s_compute));
        if (eligible) CK(cudaMemcpyAsync(c->cb_elig.p, eligible, n, cudaMemcpyHostToDevice, c->s_compute));
    }
    c->cb_n = n; c->cb_len = cb_len; c->cb_has_elig = eligible != nullptr; c->cb_resident = true;
    if (st) st->h2d_bytes += n * (size_t)cb_len * 2 + (eligible ? n : 0);
}

// the batch in c->cb_* -> c->cb_idx / c->cb_status (device); fills the device-side part of `st`
__global__ void gather_barcodes_kernel(uint32_t n, const uint32_t *__restrict__ idx, const uint8_t *__restrict__ chars, uint32_t len,
                                       uint8_t *__restrict__ out) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n) return;
    const uint8_t *src = chars + (size_t)idx[t] * len;
    for (uint32_t j = 0; j < len; j++) out[(size_t)t * len + j] = src[j];
}

static void cb_run(nb200_ctx *c, DevWhitelist &W, nb200_cb_stats *st) {
    const uint64_t n = c->cb_n;
    if (!c->cb_resident || c->cb_len != W.cb_len) throw std::runtime_error("barcode batch length does not match the whitelist");
    cudaStream_t s = c->s_compute;
    c->cb_keys.ensure(n * 8 + 16); c->cb_idx.ensure(n * 4 + 16); c->cb_status.ensure(n + 16);
    c->permA.ensure(n * 4 + 16);                        // miss list
    c->cb_inval.ensure(n * 4 + 16);
    c->flag.ensure(n + 16);                             // multi-candidate flags
    uint64_t launches = 0;
    cudaEvent_t e0 = new_event(c), e1 = new_event(c);
    CK(cudaEventRecord(e0, s));
    const size_t n_ent = W.entries.size();
    if (st) {                                           // hit flags per whitelist entry (for the cache-size statistic)
        c->cb_hit.ensure(n_ent + 16);
        CK(cudaMemsetAsync(c->cb_hit.p, 0, n_ent + 16, s));
    }
    const uint64_t launches0 = c->launches;
    cb_launch(c, W.dev, s, c->cb_chars.as<uint8_t>(), c->cb_qual.as<uint8_t>(), c->cb_has_elig ? c->cb_elig.as<uint8_t>() : nullptr, n,
              c->cb_keys.as<uint64_t>(), c->cb_idx.as<int32_t>(), c->cb_status.as<uint8_t>(), c->permA.as<uint32_t>(),
              c->cb_inval.as<uint32_t>(), (uint32_t)n, st ? c->cb_hit.as<uint8_t>() : nullptr, c->flag.as<uint8_t>(), c->d_cbctr.as<CbCounters>());
    CbCounters h{};
    if (n) {
        CK(cudaMemcpyAsync(&h, c->d_cbctr.p, sizeof h, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        if (h.n_multi) {
            // the reference's correction_cache: first read in file order decides per raw barcode
            c->permB.ensure(n * 4 + 16);
            const uint32_t m = cub_select(c, c->flag.as<uint8_t>(), c->permB.as<uint32_t>(), (uint32_t)n);   // ascending read index
            cb_first_decides(c, c->permB.as<uint32_t>(), c->cb_keys.as<uint64_t>(), m, c->cb_idx.as<int32_t>());
        }
    }
    launches += c->launches - launches0;
    uint64_t distinct = 0;
    if (st && n) {
        // "Correction cache size": distinct raw barcodes among the eligible reads = whitelist entries hit
        // exactly + distinct raw barcodes among the misses (a small sort) + distinct non-ACGTN strings
        c->num.ensure(16);
        CK(cudaMemsetAsync(c->num.p, 0, 8, s));
        cb_count_flags_kernel<<<nblk(n_ent, 256), 256, 0, s>>>(c->cb_hit.as<uint8_t>(), n_ent, c->num.as<unsigned long long>());
        const uint32_t m = (uint32_t)h.n_miss;
        if (m) {
            c->k64A.ensure((size_t)m * 8 + 16); c->k64B.ensure((size_t)m * 8 + 16);
            cb_gather_keys_kernel<<<nblk(m, 256), 256, 0, s>>>(c->permA.as<uint32_t>(), c->cb_keys.as<uint64_t>(), m, c->k64A.as<uint64_t>());
            size_t bytes = 0;
            const int bits = std::min(64, 3 * W.cb_len);
            CK(cub::DeviceRadixSort::SortKeys(nullptr, bytes, c->k64A.as<uint64_t>(), c->k64B.as<uint64_t>(), (int)m, 0, bits, s));
            c->cub_tmp.ensure(bytes);
            CK(cub::DeviceRadixSort::SortKeys(c->cub_tmp.p, bytes, c->k64A.as<uint64_t>(), c->k64B.as<uint64_t>(), (int)m, 0, bits, s));
            cb_count_distinct_kernel<<<nblk(m, 256), 256, 0, s>>>(c->k64B.as<uint64_t>(), m, c->num.as<unsigned long long>());
            launches += 8;
        }
        CK(cudaGetLastError());
        unsigned long long d = 0;
        CK(cudaMemcpyAsync(&d, c->num.p, 8, cudaMemcpyDeviceToHost, s));
        launches += 1;
        // reads with a byte outside ACGTN: distinct STRINGS, counted on the host (rare)
        std::vector<uint32_t> il;
        std::vector<char> chars;
        const uint64_t ni = h.n_inval;
        if (ni) {
            il.resize(ni);
            CK(cudaMemcpyAsync(il.data(), c->cb_inval.p, ni * 4, cudaMemcpyDeviceToHost, s));
        }
        CK(cudaStreamSynchronize(s));
        distinct = d;
        if (ni) {
            // the barcodes themselves: gathered on the device into one block, ONE copy (an input full of lowercase or '.'
            // barcodes would otherwise mean one tiny copy per read)
            chars.resize(ni * (size_t)W.cb_len);
            c->cb_inval_chars.ensure(ni * (size_t)W.cb_len + 16);
            gather_barcodes_kernel<<<nblk(ni, 256), 256, 0, s>>>((uint32_t)ni, c->cb_inval.as<uint32_t>(), c->cb_chars.as<uint8_t>(),
                                                                  (uint32_t)W.cb_len, c->cb_inval_chars.as<uint8_t>());
            launches += 1;
            CK(cudaMemcpyAsync(chars.data(), c->cb_inval_chars.p, ni * (size_t)W.cb_len, cudaMemcpyDeviceToHost, s));
            CK(cudaStreamSynchronize(s));
            std::unordered_set<std::string> seen;
            for (uint64_t t = 0; t < ni; t++) seen.emplace(chars.data() + t * (size_t)W.cb_len, (size_t)W.cb_len);
            distinct += seen.size();
        }
    }
    CK(cudaEventRecord(e1, s));
    CK(cudaStreamSynchronize(s));
    if (st) {
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        st->kernel_ms = ms;
        st->cb_perfect_match = h.perfect; st->cb_corrected = h.corrected; st->cb_no_correction = h.none;
        st->n_exact_miss = h.n_miss; st->n_multi = h.n_multi; st->probes = h.probes;
        st->cache_size = distinct; st->launches = launches;
    }
}

static void cb_fetch(nb200_ctx *c, int32_t *out_idx, uint8_t *out_status, nb200_cb_stats *st) {
    const uint64_t n = c->cb_n;
    if (n && out_idx) CK(cudaMemcpyAsync(out_idx, c->cb_idx.p, n * 4, cudaMemcpyDeviceToHost, c->s_compute));
    if (n && out_status) CK(cudaMemcpyAsync(out_status, c->cb_status.p, n, cudaMemcpyDeviceToHost, c->s_compute));
    CK(cudaStreamSynchronize(c->s_compute));
    if (st) st->d2h_bytes += (out_idx ? n * 4 : 0) + (out_status ? n : 0);
}

// Inside a catch block: the status code of the exception being handled, its message in `what`.
static int32_t status_of_exception(std::string &what) {
    try { throw; }
    catch (const IoError &e) { what = e.what(); return NB200_EIO; }
    catch (const CudaError &e) { what = e.what(); cudaGetLastError(); return NB200_ECUDA; }
    catch (const LimitError &e) { what = e.what(); return NB200_ELIMIT; }
    catch (const std::bad_alloc &) { what = "out of host memory"; return NB200_EINVAL; }
    catch (const std::exception &e) { what = e.what(); return NB200_EINVAL; }
}

}  // namespace nb200

// =============================================================================================
// C ABI
// =============================================================================================
#define API_BEGIN(ctx)                                                                             \
    if (!(ctx)) return NB200_EINVAL;                                                               \
    try {                                                                                          \
        if (cudaSetDevice((ctx)->device) != cudaSuccess) { (ctx)->err = "cudaSetDevice failed"; return NB200_ECUDA; }
#define API_END(ctx)                                                                               \
    }                                                                                              \
    catch (const std::exception &) { return nb200::status_of_exception((ctx)->err); }              \
    return NB200_OK;

extern "C" {

const char *nb200_version(void) { return "nimble_b200 0.1.0 (sm_100a)"; }

int32_t nb200_create(int32_t device, int32_t host_threads, nb200_ctx **out) {
    if (!out) return NB200_EINVAL;
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        g_create_err = std::string("no CUDA device: ") + cudaGetErrorString(e) + " (nimble_b200 has no CPU path)";
        cudaGetLastError();
        return NB200_ENODEVICE;
    }
    if (device < 0 || device >= n) { g_create_err = "device index out of range"; return NB200_EINVAL; }
    auto c = std::make_unique<nb200_ctx>();
    c->device = device;
    c->host_threads = host_threads > 0 ? host_threads : (int)std::max(1u, std::thread::hardware_concurrency());
    try {
        CK(cudaSetDevice(device));
        cudaDeviceProp p;
        CK(cudaGetDeviceProperties(&p, device));
        c->sm_count = p.multiProcessorCount;
        CK(cudaStreamCreateWithFlags(&c->s_compute.h, cudaStreamNonBlocking));
        // highest priority: the copy streams also run the tiny record-expansion kernels of the compact wire form, so that
        // they get an SM slot as soon as a block of the running probe kernel retires and never hold up the DMA queue; s_tail
        // runs each batch's latency-bound tail beside the next batch's probe
        int least = 0, greatest = 0;
        CK(cudaDeviceGetStreamPriorityRange(&least, &greatest));
        for (Stream *s : {&c->s_copy[0], &c->s_copy[1], &c->s_tail}) CK(cudaStreamCreateWithPriority(&s->h, cudaStreamNonBlocking, greatest));
        auto counters = [](DevBuf &b, size_t bytes) { CK(cudaMalloc(&b.p, bytes)); b.cap = bytes; CK(cudaMemset(b.p, 0, bytes)); };
        counters(c->d_ctr, sizeof(Counters) + 64);
        counters(c->d_ctr_odd, sizeof(Counters) + 64);
        counters(c->d_cbctr, sizeof(CbCounters) + 64);
        c->bb[0].ctr = c->d_ctr.as<Counters>();
        c->bb[1].ctr = c->d_ctr_odd.as<Counters>();
        for (auto &b : c->bb) { CK(cudaEventCreateWithFlags(&b.tail_done.h, cudaEventDisableTiming)); CK(cudaEventCreateWithFlags(&b.probe_done.h, cudaEventDisableTiming)); }
        if (const char *e = getenv("NB200_OVERLAP")) c->overlap = atoi(e) != 0;
        c->l2_persist_max = (size_t)std::max(0, p.persistingL2CacheMaxSize);
        c->l2_window_max = (size_t)std::max(0, p.accessPolicyMaxWindowSize);
        if (c->l2_persist_max && cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, c->l2_persist_max) != cudaSuccess) {
            cudaGetLastError();
            c->l2_persist_max = 0;
        }
    } catch (const std::exception &ex) {
        g_create_err = ex.what();
        return NB200_ECUDA;
    }
    *out = c.release();
    return NB200_OK;
}

void nb200_destroy(nb200_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    delete c;                      // every buffer, pinned buffer, event and stream frees itself, with c's device current
}

const char *nb200_last_error(const nb200_ctx *c) { return c ? c->err.c_str() : g_create_err.c_str(); }

// a library built in memory: installed as a freshly built JSON library is
static void install_built(nb200_ctx *c, const HostLibrary &h, int32_t *lib_id) {
    const ImageLayout lay = image_layout(h);
    install_library({c}, h, lay, [&](uint64_t a, uint64_t n, uint8_t *dst) { image_fill(h, lay, a, n, dst); }, nullptr, "(memory)", 0.0, lib_id);
}

int32_t nb200_load_library(nb200_ctx *c, const char *json_path, const char *strand_filter, int32_t k, int32_t *lib_id) {
    API_BEGIN(c)
    load_library_path({c}, json_path, strand_filter, k, c->host_threads, lib_id);
    API_END(c)
}

int32_t nb200_load_library_mem(nb200_ctx *c, int32_t n_refs, const char *const *names, const char *const *seqs,
                               const char *const *features, const nb200_config *cfg, int32_t *lib_id) {
    API_BEGIN(c)
    if (n_refs <= 0 || !names || !seqs || !cfg) throw std::runtime_error("bad arguments");
    std::vector<std::string> n(n_refs), s(n_refs), f(n_refs);
    for (int i = 0; i < n_refs; i++) { n[i] = names[i]; s[i] = seqs[i]; f[i] = features ? features[i] : names[i]; }
    HostLibrary h;
    build_library(n, s, f, *cfg, c->host_threads, h);
    install_built(c, h, lib_id);
    API_END(c)
}

int32_t nb200_load_feature_names(nb200_ctx *c, int32_t n, const char *const *names, int32_t *lib_id) {
    API_BEGIN(c)
    if (n < 0 || (n && !names)) throw std::runtime_error("bad arguments");
    std::vector<std::string> v(n);
    for (int i = 0; i < n; i++) v[i] = names[i];
    HostLibrary h;
    build_feature_dictionary(v, h);
    install_built(c, h, lib_id);
    API_END(c)
}

static DevLibrary &get_lib(const nb200_ctx *c, int32_t id) {
    if (id < 0 || id >= (int32_t)c->libs.size()) throw std::runtime_error("bad library id");
    return *c->libs[id];
}

int32_t nb200_library_config(const nb200_ctx *cc, int32_t lib_id, nb200_config *out) {
    nb200_ctx *c = const_cast<nb200_ctx *>(cc);
    API_BEGIN(c)
    if (!out) throw std::runtime_error("out is null");
    *out = get_lib(c, lib_id).host.cfg;
    API_END(c)
}

int32_t nb200_library_set_config(nb200_ctx *c, int32_t lib_id, const nb200_config *cfg) {
    API_BEGIN(c)
    if (!cfg) throw std::runtime_error("cfg is null");
    DevLibrary &L = get_lib(c, lib_id);
    if (cfg->k != L.host.cfg.k) throw std::runtime_error("k is fixed once the index is built");
    if (cfg->max_hits_to_report < 1 || cfg->max_hits_to_report > 64) throw LimitError("max_hits_to_report must be in 1..64");
    if (cfg->strand_filter < 0 || cfg->strand_filter > 3) throw std::runtime_error("bad strand_filter");
    L.host.cfg = *cfg;
    API_END(c)
}

int32_t nb200_library_set_trim(nb200_ctx *c, int32_t lib_id, int32_t target_length, double strictness) {
    API_BEGIN(c)
    DevLibrary &L = get_lib(c, lib_id);
    if (target_length < 0) { L.host.trim_on = false; return NB200_OK; }
    if (!(strictness >= 0.0 && strictness <= 1.0) || target_length > 100000) throw std::runtime_error("trim: strictness must be in 0..1");
    L.host.trim_on = true; L.host.trim_target = target_length; L.host.trim_strictness = strictness;
    API_END(c)
}

uint32_t nb200_trim_maxinfo(const uint8_t *qual, uint32_t n, int32_t phred_offset, int32_t target_length, double strictness) {
    if (!qual || !n) return 0;
    TrimTable t;
    t.init(target_length, strictness);
    return t.keep(qual, n, phred_offset, false);
}

int32_t nb200_library_info(const nb200_ctx *cc, int32_t lib_id, int64_t *n_refs, int64_t *n_features, int64_t *n_kmers,
                           int64_t *n_classes, int64_t *table_bytes) {
    nb200_ctx *c = const_cast<nb200_ctx *>(cc);
    API_BEGIN(c)
    DevLibrary &L = get_lib(c, lib_id);
    if (n_refs) *n_refs = L.host.n_refs;
    if (n_features) *n_features = L.host.n_features;
    if (n_kmers) *n_kmers = (int64_t)L.host.n_kmers;
    if (n_classes) *n_classes = (int64_t)L.host.n_classes;
    if (table_bytes) *table_bytes = (int64_t)L.table_bytes;
    API_END(c)
}

const char *nb200_feature_name(const nb200_ctx *c, int32_t lib_id, uint32_t fid) {
    if (!c || lib_id < 0 || lib_id >= (int32_t)c->libs.size()) return nullptr;
    const auto &v = c->libs[lib_id]->host.feature_names;
    return fid < v.size() ? v[fid].c_str() : nullptr;
}

int32_t nb200_host_index_stats(const char *json_path, const char *strand_filter, int32_t k, int64_t *out6) {
    // host-only: parse + build the index images, no CUDA call (used by the CPU test-suite)
    if (!json_path || !out6) return NB200_EINVAL;
    try {
        int sf = parse_strand_filter(strand_filter);
        if (sf < 0) { g_create_err = "unknown --strand_filter value"; return NB200_EINVAL; }
        std::vector<std::string> names, seqs, feats;
        nb200_config cfg{};
        parse_library_json(json_path, names, seqs, feats, cfg);
        cfg.k = k > 0 ? k : 20;
        cfg.strand_filter = sf;
        HostLibrary L;
        build_library(names, seqs, feats, cfg, (int)std::max(1u, std::thread::hardware_concurrency()), L, /*verify=*/true);
        out6[0] = L.n_refs; out6[1] = L.n_features; out6[2] = (int64_t)L.n_kmers; out6[3] = (int64_t)L.n_classes;
        out6[4] = (int64_t)(2 * L.n_buckets); out6[5] = L.identity_features ? 1 : 0;
    } catch (const LimitError &e) { g_create_err = e.what(); return NB200_ELIMIT; }
    catch (const std::exception &e) { g_create_err = e.what(); return NB200_EINVAL; }
    return NB200_OK;
}

int32_t nb200_index_write(const char *json_path, int32_t k, int32_t host_threads, const char *out_path) {
    // host-only: the index of nb200_load_library, written as an index file (library.hpp) that loads without a build
    if (!json_path || !out_path) { g_create_err = "bad arguments"; return NB200_EINVAL; }
    try {
        if (is_index_file(json_path)) throw std::runtime_error(std::string(json_path) + " is an index file already; index takes a library JSON");
        std::vector<std::string> names, seqs, feats;
        nb200_config cfg{};
        parse_library_json(json_path, names, seqs, feats, cfg);
        cfg.k = k > 0 ? k : 20;
        const int T = host_threads > 0 ? host_threads : (int)std::max(1u, std::thread::hardware_concurrency());
        HostLibrary L;
        build_library(names, seqs, feats, cfg, T, L, getenv("NB200_VERIFY_TABLE") != nullptr);
        write_index_file(L, json_path, out_path, T);
    } catch (const std::exception &) { return status_of_exception(g_create_err); }
    return NB200_OK;
}

int32_t nb200_index_info(const char *path, int32_t verify, int64_t *out9) {
    if (!path || !out9) { g_create_err = "bad arguments"; return NB200_EINVAL; }
    try {
        IndexFile f;
        HostLibrary meta;
        open_index_file(path, f, meta);
        if (verify) verify_index_file(f, meta, (int)std::max(1u, std::thread::hardware_concurrency()));
        out9[0] = f.h.version; out9[1] = meta.cfg.k;
        out9[2] = meta.n_refs; out9[3] = meta.n_features; out9[4] = (int64_t)meta.n_kmers; out9[5] = (int64_t)meta.n_classes;
        out9[6] = (int64_t)(2 * meta.n_buckets); out9[7] = meta.identity_features ? 1 : 0; out9[8] = (int64_t)f.h.sec[kSecImage].bytes;
    } catch (const std::exception &) { return status_of_exception(g_create_err); }
    return NB200_OK;
}

int32_t nb200_host_ingest_stats(const char *const *inputs, int32_t n_inputs, int32_t threads, uint64_t *out6) {
    if (!inputs || n_inputs < 1 || n_inputs > 2 || !out6) return NB200_EINVAL;
    try {
        // the streaming reader of nb200_align_files without a device stage (no CUDA call)
        FileJob job;
        for (int i = 0; i < n_inputs; i++) job.inputs.emplace_back(inputs[i]);
        job.host_threads = threads > 0 ? threads : (int)std::max(1u, std::thread::hardware_concurrency());
        FileStats st;
        run_file_pipeline(job, &st);
        out6[0] = st.n_reads; out6[1] = st.paired ? 1 : 0; out6[2] = st.has_tags ? 1 : 0;
        out6[3] = st.bases1; out6[4] = st.bases2; out6[5] = st.checksum;
    } catch (const IoError &e) { g_create_err = e.what(); return NB200_EIO; }
    catch (const std::exception &e) { g_create_err = e.what(); return NB200_EINVAL; }
    return NB200_OK;
}

int32_t nb200_pack_layout(uint32_t max_len, uint32_t *words, uint32_t *stride) {
    if (max_len > NB200_MAX_READ_LEN) return NB200_EINVAL;
    uint32_t w = (max_len + 31) / 32;
    if (w == 0) w = 1;
    if (words) *words = w;
    if (stride) *stride = (12 * w + 15) & ~15u;
    return NB200_OK;
}

int32_t nb200_pack_reads(nb200_ctx *c, const char *bases, const int64_t *off, uint64_t n, uint32_t words, uint32_t stride,
                         uint8_t *out, uint16_t *out_len) {
    if (!bases || !off || !out || !out_len || words == 0 || stride < 12 * words) return NB200_EINVAL;
    const int T = c ? c->host_threads : (int)std::max(1u, std::thread::hardware_concurrency());
    std::atomic<int> bad{0};
    uint8_t lut[256];
    memset(lut, 4, sizeof lut);
    lut['A'] = lut['a'] = 0; lut['C'] = lut['c'] = 1; lut['G'] = lut['g'] = 2; lut['T'] = lut['t'] = 3;
    auto work = [&](uint64_t a, uint64_t b) {
        for (uint64_t i = a; i < b; i++) {
            const int64_t L = off[i + 1] - off[i];
            if (L < 0 || L > (int64_t)words * 32 || L > NB200_MAX_READ_LEN) { bad = 1; out_len[i] = 0; continue; }
            uint8_t *rec = out + i * (size_t)stride;
            uint64_t *seq = reinterpret_cast<uint64_t *>(rec);
            uint32_t *nm = reinterpret_cast<uint32_t *>(rec + (size_t)words * 8);
            const unsigned char *s = reinterpret_cast<const unsigned char *>(bases + off[i]);
            // 32 bases per output word, accumulated in registers; lut: bits 0-1 code, bit 2 = not ACGT
            int64_t j = 0;
            for (uint32_t w = 0; w < words; w++) {
                uint64_t acc = 0;
                uint32_t nacc = 0;
                const int64_t e = std::min<int64_t>(L, j + 32);
                for (int sh = 0; j < e; j++, sh++) {
                    const uint32_t v = lut[s[j]];
                    acc |= (uint64_t)(v & 3u) << (2 * sh);
                    nacc |= (v >> 2) << sh;
                }
                seq[w] = acc; nm[w] = nacc;
            }
            for (size_t t = (size_t)words * 12; t < stride; t++) rec[t] = 0;     // padding of the record
            out_len[i] = (uint16_t)L;
        }
    };
    if (T <= 1 || n < 4096) work(0, n);
    else {
        std::vector<std::thread> th;
        const uint64_t per = (n + T - 1) / T;
        for (int t = 0; t < T; t++) {
            uint64_t a = t * per, b = std::min<uint64_t>(n, a + per);
            if (a < b) th.emplace_back(work, a, b);
        }
        for (auto &x : th) x.join();
    }
    if (bad) { if (c) c->err = "read longer than the packed layout / 500 bases"; return NB200_EINVAL; }
    return NB200_OK;
}

int32_t nb200_pack_reads_compact(nb200_ctx *c, const char *bases, const int64_t *off, uint64_t n, uint32_t words, uint8_t *out,
                                 uint16_t *out_len, uint32_t *out_n_idx, uint32_t *out_n_mask, uint64_t cap, uint64_t *n_with_n) {
    if (!bases || !off || !out || !out_len || !n_with_n || words == 0 || n > 0xFFFFFFFFull) return NB200_EINVAL;
    if (cap && (!out_n_idx || !out_n_mask)) return NB200_EINVAL;
    const int T = c ? c->host_threads : (int)std::max(1u, std::thread::hardware_concurrency());
    std::atomic<int> bad{0};
    uint8_t lut[256];
    memset(lut, 4, sizeof lut);
    lut['A'] = lut['a'] = 0; lut['C'] = lut['c'] = 1; lut['G'] = lut['g'] = 2; lut['T'] = lut['t'] = 3;
    const int parts = (T <= 1 || n < 4096) ? 1 : T;
    const uint64_t per = (n + parts - 1) / std::max(1, parts);
    // reads with a non-ACGT base are rare: every thread keeps its own (index, mask words) list, joined in order below
    std::vector<std::vector<uint32_t>> side((size_t)parts);
    auto work = [&](int t) {
        const uint64_t a = (uint64_t)t * per, b = std::min<uint64_t>(n, a + per);
        std::vector<uint32_t> &sd = side[(size_t)t];
        uint32_t nm[(NB200_MAX_READ_LEN + 31) / 32];
        for (uint64_t i = a; i < b; i++) {
            const int64_t L = off[i + 1] - off[i];
            uint64_t *seq = reinterpret_cast<uint64_t *>(out + i * (size_t)words * 8);
            if (L < 0 || L > (int64_t)words * 32 || L > NB200_MAX_READ_LEN) { bad = 1; out_len[i] = 0; for (uint32_t w = 0; w < words; w++) seq[w] = 0; continue; }
            const unsigned char *s = reinterpret_cast<const unsigned char *>(bases + off[i]);
            int64_t j = 0;
            uint32_t any = 0;
            for (uint32_t w = 0; w < words; w++) {
                uint64_t acc = 0;
                uint32_t nacc = 0;
                const int64_t e = std::min<int64_t>(L, j + 32);
                for (int sh = 0; j < e; j++, sh++) {
                    const uint32_t v = lut[s[j]];
                    acc |= (uint64_t)(v & 3u) << (2 * sh);
                    nacc |= (v >> 2) << sh;
                }
                seq[w] = acc; nm[w] = nacc; any |= nacc;
            }
            out_len[i] = (uint16_t)L;
            if (any) { sd.push_back((uint32_t)i); sd.insert(sd.end(), nm, nm + words); }
        }
    };
    if (parts == 1) work(0);
    else {
        std::vector<std::thread> th;
        for (int t = 0; t < parts; t++) th.emplace_back(work, t);
        for (auto &x : th) x.join();
    }
    if (bad) { if (c) c->err = "read longer than the packed layout / 500 bases"; return NB200_EINVAL; }
    uint64_t total = 0;
    for (auto &sd : side) total += sd.size() / (words + 1);
    *n_with_n = total;
    if (total > cap) { if (c) c->err = "N side table too small"; return NB200_ELIMIT; }
    uint64_t at = 0;
    for (auto &sd : side)
        for (size_t q = 0; q < sd.size(); q += words + 1, at++) {
            out_n_idx[at] = sd[q];
            memcpy(out_n_mask + at * words, &sd[q + 1], (size_t)words * 4);
        }
    return NB200_OK;
}

int32_t nb200_pack_barcodes(const char *cb, uint32_t cb_len, const char *ub, uint32_t ub_len, uint64_t n, uint64_t *out_key) {
    if (!cb || !ub || !out_key || cb_len == 0 || cb_len > 16 || ub_len == 0 || ub_len > 16) return NB200_EINVAL;
    for (uint64_t i = 0; i < n; i++) {
        uint64_t a = 0, b = 0;
        bool ok = true;
        for (uint32_t j = 0; j < cb_len && ok; j++) {
            switch (cb[i * cb_len + j]) {
            case 'A': a = a << 2; break; case 'C': a = (a << 2) | 1; break;
            case 'G': a = (a << 2) | 2; break; case 'T': a = (a << 2) | 3; break;
            default: ok = false;
            }
        }
        for (uint32_t j = 0; j < ub_len && ok; j++) {
            switch (ub[i * ub_len + j]) {
            case 'A': b = b << 2; break; case 'C': b = (b << 2) | 1; break;
            case 'G': b = (b << 2) | 2; break; case 'T': b = (b << 2) | 3; break;
            default: ok = false;
            }
        }
        out_key[i] = ok ? ((a << 32) | b) : NB200_NO_BARCODE;
    }
    return NB200_OK;
}

void *nb200_alloc_pinned(size_t bytes) {
    void *p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
void nb200_free_pinned(void *p) { if (p) cudaFreeHost(p); }

int32_t nb200_upload(nb200_ctx *c, const nb200_reads *r1, const nb200_reads *r2, const uint64_t *key) {
    API_BEGIN(c)
    if (!r1) throw std::runtime_error("r1 is null");
    validate_reads(r1, "r1");
    if (r2) { validate_reads(r2, "r2"); if (r2->n != r1->n) throw std::runtime_error("r1 and r2 differ in read count"); }
    ensure_read_buffers(c, r1, r2, key != nullptr);
    h2d_reads(c, c->s_compute, r1, c->stage1, c->d_r1.as<uint8_t>(), c->d_r1len.as<uint16_t>(), 0, r1->n);
    if (r2) h2d_reads(c, c->s_compute, r2, c->stage2, c->d_r2.as<uint8_t>(), c->d_r2len.as<uint16_t>(), 0, r2->n);
    if (key) CK(cudaMemcpyAsync(c->d_key.p, key, r1->n * 8, cudaMemcpyHostToDevice, c->s_compute));
    CK(cudaStreamSynchronize(c->s_compute));
    c->resident = true;
    API_END(c)
}

// The flags word of the counting entries (NB200_UMI_*).  may_correct = false where keys are caller-assigned ids rather
// than UMI codes (nb200_align, nb200_align_resident).
static int32_t check_umi_flags(int32_t flags, bool may_correct) {
    if (flags & ~(NB200_UMI_NO_THRESHOLD | NB200_UMI_CORRECT)) throw std::runtime_error("unknown bits in the UMI flags word");
    if (!may_correct && (flags & NB200_UMI_CORRECT))
        throw std::runtime_error("NB200_UMI_CORRECT needs UMIs as sequence codes: use the file or report entries");
    return flags;
}

int32_t nb200_align_resident(nb200_ctx *c, int32_t lib_id, double umi_threshold, int32_t disable_thresholding,
                             nb200_counts *counts) {
    API_BEGIN(c)
    if (!counts) throw std::runtime_error("counts is null");
    check_umi_flags(disable_thresholding, false);
    if (!c->resident) throw std::runtime_error("no resident reads: call nb200_upload first");
    run_align(c, get_lib(c, lib_id), nullptr, umi_threshold, disable_thresholding, counts);
    API_END(c)
}

int32_t nb200_umi_neighbours(uint32_t code, uint32_t *out_code, uint32_t *out_value) {
    if (!out_code || !out_value) return NB200_EINVAL;
    if (code < 1 || code > kUmiCodeMax) return -1;
    int n = 0;
    umi_for_each_neighbour(code, umi_byte_value(code), [&](uint32_t v, uint32_t bv) { out_code[n] = v; out_value[n] = bv; n++; });
    return n;
}

int32_t nb200_umis_corrected(const nb200_ctx *c, uint64_t *out) {
    if (!c || !out) return NB200_EINVAL;
    *out = c->umis_corrected;
    return NB200_OK;
}

int32_t nb200_counts_device(const nb200_ctx *c, uint64_t *n_rows, uint64_t *n_ids, const uint32_t **cell, const uint32_t **count,
                            const uint32_t **feat_off, const uint32_t **feat_ids) {
    if (!c || !n_rows || !n_ids || !cell || !count || !feat_off || !feat_ids) return NB200_EINVAL;
    *n_rows = c->dev_rows; *n_ids = c->dev_ids;
    *cell = c->o_cell_d.as<uint32_t>(); *count = c->o_count_d.as<uint32_t>();
    *feat_off = c->o_off_d.as<uint32_t>(); *feat_ids = c->o_ids_d.as<uint32_t>();
    return NB200_OK;
}

int32_t nb200_fetch_results(nb200_ctx *c, nb200_read_result *results, int32_t *feats) {
    API_BEGIN(c)
    if (results) CK(cudaMemcpy(results, c->results.p, c->n_reads * sizeof(nb200_read_result), cudaMemcpyDeviceToHost));
    if (feats) CK(cudaMemcpy(feats, c->feats.p, c->n_reads * (size_t)c->feats_stride * 4, cudaMemcpyDeviceToHost));
    API_END(c)
}

int32_t nb200_align(nb200_ctx *c, int32_t lib_id, const nb200_reads *r1, const nb200_reads *r2, const uint64_t *key,
                    double umi_threshold, int32_t disable_thresholding, nb200_read_result *results, int32_t *feats,
                    nb200_counts *counts) {
    API_BEGIN(c)
    if (!r1 || !counts) throw std::runtime_error("r1 / counts is null");
    check_umi_flags(disable_thresholding, false);
    validate_reads(r1, "r1");
    if (r2) { validate_reads(r2, "r2"); if (r2->n != r1->n) throw std::runtime_error("r1 and r2 differ in read count"); }
    ensure_read_buffers(c, r1, r2, key != nullptr);
    HostInput in{r1, r2, key};
    run_align(c, get_lib(c, lib_id), &in, umi_threshold, disable_thresholding, counts);
    c->resident = true;
    if (results) {
        CK(cudaMemcpy(results, c->results.p, r1->n * sizeof(nb200_read_result), cudaMemcpyDeviceToHost));
        c->timing.d2h_bytes += r1->n * sizeof(nb200_read_result);
    }
    if (feats) {
        CK(cudaMemcpy(feats, c->feats.p, r1->n * (size_t)c->feats_stride * 4, cudaMemcpyDeviceToHost));
        c->timing.d2h_bytes += r1->n * (size_t)c->feats_stride * 4;
    }
    API_END(c)
}

// reads in memory (the 10x one-pass route) -> per library: GPU path -> per-read TSV
static void align_readset(nb200_ctx *c, const ReadSet &R, const int32_t *lib_ids, const char *const *outputs, int32_t n_libs,
                          PhaseTimer &pt) {
    const uint64_t n = R.r1.size();
    auto pack = [&](const Arena &a, std::vector<uint8_t> &buf, std::vector<uint16_t> &len, nb200_reads &out) {
        int64_t ml = 1;
        for (uint64_t i = 0; i < n; i++) ml = std::max<int64_t>(ml, a.off[i + 1] - a.off[i]);
        if (ml > NB200_MAX_READ_LEN) throw std::runtime_error("read longer than 500 bases");
        uint32_t words, stride;
        nb200_pack_layout((uint32_t)ml, &words, &stride);
        buf.assign(n * (size_t)stride + 64, 0); len.assign(n + 1, 0);
        if (n && nb200_pack_reads(c, a.data.data(), a.off.data(), n, words, stride, buf.data(), len.data()) != 0)
            throw std::runtime_error(c->err);
        out = nb200_reads{buf.data(), len.data(), n, stride, words};
    };
    std::vector<uint8_t> b1, b2;
    std::vector<uint16_t> l1, l2;
    nb200_reads p1{}, p2{};
    pack(R.r1, b1, l1, p1);
    pack(R.r2, b2, l2, p2);
    pt.lap("2-bit pack");
    for (int li = 0; li < n_libs; li++) {
        DevLibrary &L = get_lib(c, lib_ids[li]);
        const int mh = L.host.cfg.max_hits_to_report;
        std::vector<nb200_read_result> res(n + 1);
        std::vector<int32_t> feats((n + 1) * (size_t)mh);
        nb200_counts counts{};
        ensure_read_buffers(c, &p1, &p2, false);
        HostInput hin{&p1, &p2, nullptr};
        run_align(c, L, &hin, 0.05, 0, &counts);
        c->resident = true;
        pt.lap("GPU align");
        if (n) {
            CK(cudaMemcpy(res.data(), c->results.p, n * sizeof(nb200_read_result), cudaMemcpyDeviceToHost));
            CK(cudaMemcpy(feats.data(), c->feats.p, n * (size_t)mh * 4, cudaMemcpyDeviceToHost));
        }
        pt.lap("fetch per-read results");
        write_per_read_tsv(outputs[li], R, res.data(), feats.data(), mh, L.host.feature_names, c->host_threads);
        pt.lap("write TSV");
    }
}

// values per library in the out3 of the counting entries: rows used, count rows written, UMIs dropped (+ UMIs corrected)
static int out3_per_lib(int32_t umi_flags) { return (umi_flags & NB200_UMI_CORRECT) ? 4 : 3; }

// File-level entries: what the aligner process does between its argv and its exit code (nimble/__main__.py:177-196),
// streaming (stream.cpp).  One pass over `inputs` on the contexts `ctxs`, whose libraries carry the same ids in the same
// order; per library a per-read TSV (outputs) and/or a counts TSV (counts_outputs).  whitelist: the 10x mode of
// fastq-to-counts (inputs = raw R1 and R2), null otherwise.
static FileStats run_job(const std::vector<nb200_ctx *> &ctxs, const int32_t *lib_ids, int32_t n_libs, const char *const *inputs,
                         int32_t n_inputs, const char *const *outputs, const char *const *counts_outputs, double umi_threshold,
                         int32_t disable_thresholding, const char *whitelist, int32_t cb_len, int32_t umi_len) {
    FileJob job;
    std::vector<std::string> wl;
    if (whitelist) { read_whitelist_lines(whitelist, wl); job.whitelist = &wl; job.cb_len = cb_len; job.umi_len = umi_len; }
    job.inputs.assign(inputs, inputs + n_inputs);
    job.ctxs = ctxs;
    job.lib_ids.assign(lib_ids, lib_ids + n_libs);
    for (int i = 0; i < n_libs; i++) {
        get_lib(ctxs[0], lib_ids[i]);
        if (outputs) job.outputs.emplace_back(outputs[i]);
        if (counts_outputs) job.counts_outputs.emplace_back(counts_outputs[i]);
    }
    job.host_threads = ctxs[0]->host_threads;
    job.umi_threshold = umi_threshold;
    job.umi_flags = disable_thresholding;
    FileStats st;
    run_file_pipeline(job, &st);
    if (getenv("NB200_TRACE"))
        fprintf(stderr, "[nb200 trace] file pipeline: %llu reads in %llu slabs on %zu GPUs, %.3f s (%.2f M reads/s), %d host threads\n",
                (unsigned long long)st.n_reads, (unsigned long long)st.n_slabs, ctxs.size(), st.seconds,
                st.n_reads / std::max(st.seconds, 1e-9) / 1e6, job.host_threads);
    return st;
}

int32_t nb200_align_files(nb200_ctx *c, const char *const *inputs, int32_t n_inputs, const int32_t *lib_ids,
                          const char *const *outputs, int32_t n_libs) {
    API_BEGIN(c)
    if (!inputs || n_inputs < 1 || n_inputs > 2 || !lib_ids || !outputs || n_libs < 1) throw std::runtime_error("bad arguments");
    run_job({c}, lib_ids, n_libs, inputs, n_inputs, outputs, nullptr, 0.05, 0, nullptr, 0, 0);
    API_END(c)
}

// The same pipeline over several GPUs of one node, in ONE process: libraries are loaded on every device (index
// replicated), the reader deals slabs of reads to whichever GPU has a free lane, the writer restores input order
// (SURVEY.md §8e: reads are independent up to the per-read TSV).  With counts outputs the rows of the UMI stage stay in
// each device's row store and are gathered on the first device at the end (lane_rows_count).
static int32_t files_multi(const int32_t *devices, int32_t n_devices, int32_t host_threads, const char *const *inputs, int32_t n_inputs,
                           const char *const *library_json, int32_t n_libs, const char *strand_filter, int32_t k, const char *trim,
                           const char *const *outputs, const char *const *counts_outputs, double umi_threshold, int32_t disable_thresholding,
                           uint64_t *out3, char *err, size_t err_cap, double *stats4, const char *whitelist = nullptr, int32_t cb_len = 16,
                           int32_t umi_len = 12, nb200_cb_stats *cb_stats = nullptr);

int32_t nb200_align_files_multi(const int32_t *devices, int32_t n_devices, int32_t host_threads, const char *const *inputs, int32_t n_inputs,
                                const char *const *library_json, int32_t n_libs, const char *strand_filter, int32_t k,
                                const char *const *outputs, const char *trim, char *err, size_t err_cap, double *stats4) {
    if (!outputs) { if (err && err_cap) snprintf(err, err_cap, "bad arguments"); return NB200_EINVAL; }
    return files_multi(devices, n_devices, host_threads, inputs, n_inputs, library_json, n_libs, strand_filter, k, trim, outputs, nullptr,
                       0.0, 0, nullptr, err, err_cap, stats4);
}

int32_t nb200_align_files_counts_multi(const int32_t *devices, int32_t n_devices, int32_t host_threads,
                                       const char *const *inputs, int32_t n_inputs, const char *const *library_json,
                                       int32_t n_libs, const char *strand_filter, int32_t k, const char *trim,
                                       const char *const *per_read_outputs, const char *const *counts_outputs,
                                       double umi_threshold, int32_t disable_thresholding,
                                       uint64_t *out3, char *err, size_t err_cap, double *stats4) {
    if (!counts_outputs) { if (err && err_cap) snprintf(err, err_cap, "bad arguments"); return NB200_EINVAL; }
    return files_multi(devices, n_devices, host_threads, inputs, n_inputs, library_json, n_libs, strand_filter, k, trim, per_read_outputs,
                       counts_outputs, umi_threshold, disable_thresholding, out3, err, err_cap, stats4);
}

int32_t nb200_align_files_counts(nb200_ctx *c, const char *const *inputs, int32_t n_inputs, const int32_t *lib_ids,
                                 const char *const *per_read_outputs, const char *const *counts_outputs, int32_t n_libs,
                                 double umi_threshold, int32_t disable_thresholding, uint64_t *out3) {
    API_BEGIN(c)
    if (!inputs || n_inputs < 1 || n_inputs > 2 || !lib_ids || !counts_outputs || n_libs < 1) throw std::runtime_error("bad arguments");
    check_umi_flags(disable_thresholding, true);
    if (out3) for (int i = 0; i < out3_per_lib(disable_thresholding) * n_libs; i++) out3[i] = 0;
    const FileStats st = run_job({c}, lib_ids, n_libs, inputs, n_inputs, per_read_outputs, counts_outputs, umi_threshold,
                                 disable_thresholding, nullptr, 0, 0);
    if (out3) for (size_t i = 0; i < st.counts3.size(); i++) out3[i] = st.counts3[i];
    API_END(c)
}

static int32_t files_multi(const int32_t *devices, int32_t n_devices, int32_t host_threads, const char *const *inputs, int32_t n_inputs,
                           const char *const *library_json, int32_t n_libs, const char *strand_filter, int32_t k, const char *trim,
                           const char *const *outputs, const char *const *counts_outputs, double umi_threshold, int32_t disable_thresholding,
                           uint64_t *out3, char *err, size_t err_cap, double *stats4, const char *whitelist, int32_t cb_len,
                           int32_t umi_len, nb200_cb_stats *cb_stats) {
    auto fail = [&](int32_t rc, const std::string &w) { if (err && err_cap) { snprintf(err, err_cap, "%s", w.c_str()); } return rc; };
    if (!devices || n_devices < 1 || !inputs || n_inputs < 1 || n_inputs > 2 || !library_json || n_libs < 1 || (!outputs && !counts_outputs))
        return fail(NB200_EINVAL, "bad arguments");
    try { check_umi_flags(disable_thresholding, true); } catch (const std::exception &e) { return fail(NB200_EINVAL, e.what()); }
    if (out3 && counts_outputs) for (int i = 0; i < out3_per_lib(disable_thresholding) * n_libs; i++) out3[i] = 0;
    std::vector<std::pair<int, double>> trims;
    try { trims = parse_trim_arg(trim, (size_t)n_libs); } catch (const std::exception &e) { return fail(NB200_EINVAL, e.what()); }
    std::vector<nb200_ctx *> ctxs;
    int32_t rc = NB200_OK;
    std::string what;
    for (int d = 0; d < n_devices && rc == NB200_OK; d++) {
        nb200_ctx *c = nullptr;
        rc = nb200_create(devices[d], host_threads, &c);
        if (rc != NB200_OK) { what = nb200_last_error(nullptr); break; }
        ctxs.push_back(c);
    }
    std::vector<int32_t> ids(n_libs, -1);
    if (rc == NB200_OK) {
        // each library built (or its index file read) once, its image copied to every device
        try {
            for (int li = 0; li < n_libs; li++) {
                load_library_path(ctxs, library_json[li], strand_filter, k, ctxs[0]->host_threads, &ids[li]);
                if (!trims.empty())
                    for (nb200_ctx *c : ctxs) {
                        rc = nb200_library_set_trim(c, ids[li], trims[(size_t)li].first, trims[(size_t)li].second);
                        if (rc != NB200_OK) { what = nb200_last_error(c); break; }
                    }
                if (rc != NB200_OK) break;
            }
        } catch (const std::exception &) { rc = status_of_exception(what); }
    }
    if (rc == NB200_OK) {
        try {
            const FileStats st = run_job(ctxs, ids.data(), n_libs, inputs, n_inputs, outputs, counts_outputs, umi_threshold,
                                         disable_thresholding, whitelist, cb_len, umi_len);
            if (stats4) { stats4[0] = (double)st.n_reads; stats4[1] = st.seconds; stats4[2] = (double)st.called; stats4[3] = (double)st.n_slabs; }
            if (out3) for (size_t i = 0; i < st.counts3.size(); i++) out3[i] = st.counts3[i];
            if (cb_stats) *cb_stats = st.cb;
        } catch (const std::exception &) { rc = status_of_exception(what); }
    }
    for (nb200_ctx *c : ctxs) nb200_destroy(c);
    return rc == NB200_OK ? NB200_OK : fail(rc, what);
}

// fastq-to-bam + align --counts without the intermediate BAM, streaming (stream.cpp, 10x mode): one pass from raw R1 / R2
// to the counts TSVs, the cell barcodes corrected slab by slab on the device, the correction cache over the whole call.
int32_t nb200_fastq_to_counts(nb200_ctx *c, const char *r1_fastq, const char *r2_fastq, const char *whitelist_path, int32_t cb_len,
                              int32_t umi_len, const int32_t *lib_ids, const char *const *counts_outputs, int32_t n_libs,
                              double umi_threshold, int32_t disable_thresholding, uint64_t *out3, nb200_cb_stats *stats) {
    API_BEGIN(c)
    if (!r1_fastq || !r2_fastq || !whitelist_path || !lib_ids || !counts_outputs || n_libs < 1 || cb_len < 1 || cb_len > kCbMaxLen || umi_len < 0)
        throw std::runtime_error("bad arguments");
    check_umi_flags(disable_thresholding, true);
    if (out3) for (int i = 0; i < out3_per_lib(disable_thresholding) * n_libs; i++) out3[i] = 0;
    if (stats) *stats = nb200_cb_stats{};
    const char *inputs[2] = {r1_fastq, r2_fastq};
    const FileStats st = run_job({c}, lib_ids, n_libs, inputs, 2, nullptr, counts_outputs, umi_threshold, disable_thresholding,
                                 whitelist_path, cb_len, umi_len);
    if (out3) for (size_t i = 0; i < st.counts3.size(); i++) out3[i] = st.counts3[i];
    if (stats) *stats = st.cb;
    API_END(c)
}

int32_t nb200_fastq_to_counts_multi(const int32_t *devices, int32_t n_devices, int32_t host_threads, const char *r1_fastq,
                                    const char *r2_fastq, const char *whitelist_path, int32_t cb_len, int32_t umi_len,
                                    const char *const *library_json, int32_t n_libs, const char *strand_filter, int32_t k,
                                    const char *trim, const char *const *counts_outputs, double umi_threshold,
                                    int32_t disable_thresholding, uint64_t *out3, nb200_cb_stats *stats, char *err, size_t err_cap,
                                    double *stats4) {
    if (stats) *stats = nb200_cb_stats{};
    if (!r1_fastq || !r2_fastq || !whitelist_path || !counts_outputs || cb_len < 1 || cb_len > kCbMaxLen || umi_len < 0) {
        if (err && err_cap) snprintf(err, err_cap, "bad arguments");
        return NB200_EINVAL;
    }
    const char *inputs[2] = {r1_fastq, r2_fastq};
    return files_multi(devices, n_devices, host_threads, inputs, 2, library_json, n_libs, strand_filter, k, trim, nullptr, counts_outputs,
                       umi_threshold, disable_thresholding, out3, err, err_cap, stats4, whitelist_path, cb_len, umi_len, stats);
}

// fastq-to-bam + align without the intermediate BAM: the pairs fastq_to_bam_with_barcodes would write
// (corrected CB, raw UB, read 1 = R1 minus barcode+UMI, read 2 = R2) go straight to the aligner.
int32_t nb200_align_10x_fastq(nb200_ctx *c, const char *r1_fastq, const char *r2_fastq, const char *whitelist_path, int32_t cb_len,
                              int32_t umi_len, const int32_t *lib_ids, const char *const *outputs, int32_t n_libs,
                              nb200_cb_stats *stats) {
    API_BEGIN(c)
    if (!r1_fastq || !r2_fastq || !whitelist_path || !lib_ids || !outputs || n_libs < 1 || cb_len < 1 || umi_len < 0)
        throw std::runtime_error("bad arguments");
    PhaseTimer pt;
    nb200_cb_stats st{};
    std::vector<std::string> lines;
    read_whitelist_lines(whitelist_path, lines);
    std::unique_ptr<DevWhitelist> W = build_whitelist(c, std::move(lines), cb_len);
    FastqQ A, B;
    {
        std::string err;
        std::thread t([&] { try { load_fastq_qual(r2_fastq, B); } catch (const std::exception &e) { err = e.what(); } });
        try { load_fastq_qual(r1_fastq, A); } catch (...) { t.join(); throw; }
        t.join();
        if (!err.empty()) throw IoError(err);
    }
    pt.lap("whitelist + FASTQ parse");
    const size_t n = std::min(A.recs.size(), B.recs.size());
    std::vector<uint8_t> cb(n * (size_t)cb_len + 16), qual(n * (size_t)cb_len + 16), elig(n + 16);
    slice_barcodes(A, B, cb_len, umi_len, c->host_threads, cb.data(), qual.data(), elig.data(), st);
    std::vector<int32_t> idx(n + 1);
    std::vector<uint8_t> status(n + 1);
    nb200_cb_stats dev{};
    cb_upload(c, cb_len, (const char *)cb.data(), qual.data(), elig.data(), n, &dev);
    cb_run(c, *W, &dev);
    cb_fetch(c, idx.data(), status.data(), &dev);
    c->ev_pool.clear();
    c->cb_resident = false;
    dev.total_pairs = st.total_pairs; dev.name_mismatch = st.name_mismatch; dev.too_short = st.too_short;
    dev.no_remaining_seq = st.no_remaining_seq;
    pt.lap("barcode correction");
    ReadSet R;
    const uint32_t bl = (uint32_t)(cb_len + umi_len);
    uint64_t written = 0;
    for (size_t i = 0; i < n; i++) {
        if (status[i] != NB200_CB_PERFECT && status[i] != NB200_CB_CORRECTED) continue;
        const FqRec &x = A.recs[i], &y = B.recs[i];
        const char *t1 = A.text.data(), *t2 = B.text.data();
        uint32_t nl = x.name_len;
        if (nl >= 2 && t1[x.name + nl - 2] == '/' && t1[x.name + nl - 1] == '1') nl -= 2;
        const std::string &cbs = W->entries[(size_t)idx[i]];
        R.names.add(t1 + x.name, nl);
        R.r1.add(t1 + x.seq + bl, x.len - bl);
        R.r2.add(t2 + y.seq, y.len);
        R.cb.add(cbs.data(), cbs.size());
        R.ub.add(t1 + x.seq + cb_len, (size_t)umi_len);
        written++;
    }
    dev.written_pairs = written;
    pt.lap("build read set");
    align_readset(c, R, lib_ids, outputs, n_libs, pt);
    if (stats) *stats = dev;
    API_END(c)
}

int32_t nb200_umi_counts(nb200_ctx *c, int32_t lib_id, uint64_t n_rows, const uint64_t *key, const uint32_t *off,
                         const uint32_t *feat_ids, const double *score, double umi_threshold, int32_t disable_thresholding,
                         nb200_counts *counts) {
    API_BEGIN(c)
    if (!counts || (n_rows && (!off || !key))) throw std::runtime_error("bad arguments");
    check_umi_flags(disable_thresholding, true);
    DevLibrary &L = get_lib(c, lib_id);
    uint32_t stride = 1;
    for (uint64_t i = 0; i < n_rows; i++) {
        if (off[i + 1] < off[i]) throw std::runtime_error("off is not monotone");
        stride = std::max(stride, off[i + 1] - off[i]);
    }
    if (stride > 65535) throw LimitError("a row lists more than 65535 features");
    if (n_rows > 0x7FFFFFF0ull) throw LimitError("more than 2^31 rows in one call");
    const uint64_t n_ids = n_rows ? off[n_rows] : 0;
    if (n_ids && !feat_ids) throw std::runtime_error("bad arguments");
    c->timing = nb200_timing{};
    c->launches = 0;
    // the CSR goes up as it is (4 B per id, no padding to the longest row) and the kernels read it in place
    c->gen_off.ensure((n_rows + 1) * 4 + 16); c->gen_feats.ensure(n_ids * 4 + 16); c->gen_key.ensure(n_rows * 8 + 16);
    cudaEvent_t e0 = new_event(c), e1 = new_event(c);
    CK(cudaEventRecord(e0, c->s_compute));
    CK(cudaMemsetAsync(c->d_ctr.p, 0, sizeof(Counters), c->s_compute));
    if (n_rows) {
        CK(cudaMemcpyAsync(c->gen_off.p, off, (n_rows + 1) * 4, cudaMemcpyHostToDevice, c->s_compute));
        if (n_ids) CK(cudaMemcpyAsync(c->gen_feats.p, feat_ids, n_ids * 4, cudaMemcpyHostToDevice, c->s_compute));
        CK(cudaMemcpyAsync(c->gen_key.p, key, n_rows * 8, cudaMemcpyHostToDevice, c->s_compute));
        c->num.ensure(64);
        CK(cudaMemsetAsync(c->num.p, 0, 4, c->s_compute));
        check_rows_kernel<<<nblk(n_rows, 256), 256, 0, c->s_compute>>>(n_rows, c->gen_off.as<uint32_t>(), c->gen_feats.as<uint32_t>(),
                                                                        (uint32_t)L.host.n_features, c->num.as<unsigned int>());
        c->launches++;
        unsigned int bad = 0;
        CK(cudaMemcpyAsync(&bad, c->num.p, 4, cudaMemcpyDeviceToHost, c->s_compute));
        CK(cudaStreamSynchronize(c->s_compute));
        if (bad & 1u) throw std::runtime_error("feature id out of range");
        if (bad & 2u) throw std::runtime_error("feature ids of a row must be ascending");
    }
    const double *d_score = nullptr;
    if (score && n_rows) {
        c->gen_score.ensure(n_rows * 8);
        CK(cudaMemcpyAsync(c->gen_score.p, score, n_rows * 8, cudaMemcpyHostToDevice, c->s_compute));
        d_score = c->gen_score.as<double>();
    }
    c->timing.h2d_bytes = (n_rows + 1) * 4 + n_ids * 4 + n_rows * (8 + (score ? 8 : 0));
    cudaEvent_t e_in = new_event(c);                      // rows resident and expanded: the UMI stage proper starts here
    CK(cudaEventRecord(e_in, c->s_compute));
    aggregate(c, L, n_rows, c->gen_key.as<uint64_t>(), Rows{c->gen_feats.as<int32_t>(), c->gen_off.as<uint32_t>(), nullptr, nullptr, 0}, d_score,
              stride, umi_threshold, disable_thresholding, counts);
    CK(cudaEventRecord(e1, c->s_compute));
    CK(cudaStreamSynchronize(c->s_compute));
    Counters h2;
    CK(cudaMemcpy(&h2, c->d_ctr.p, sizeof(h2), cudaMemcpyDeviceToHost));
    counts->dropped_empty = h2.dropped_empty;
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, e0, e1)); c->timing.total_ms = ms;
    CK(cudaEventElapsedTime(&ms, e_in, e1)); c->timing.agg_ms = ms;
    CK(cudaEventElapsedTime(&ms, e0, e_in)); c->timing.h2d_ms = ms;
    c->timing.launches = c->launches;
    c->ev_pool.clear();
    API_END(c)
}

int32_t nb200_report_file(nb200_ctx *c, const char *in_tsv, const char *out_tsv, double umi_threshold, int32_t disable_thresholding,
                          uint64_t *out3) {
    API_BEGIN(c)
    if (!in_tsv || !out_tsv) throw std::runtime_error("bad arguments");
    check_umi_flags(disable_thresholding, true);
    if (out3) for (int i = 0; i < out3_per_lib(disable_thresholding); i++) out3[i] = 0;
    ReportRows R;
    if (!parse_per_read_tsv(in_tsv, R, c->host_threads)) {
        write_counts_tsv(out_tsv, nullptr, R.feature_names, R.cells);       // write_empty_df
        return NB200_OK;
    }
    int32_t lib_id = -1;
    {
        HostLibrary h;
        build_feature_dictionary(R.feature_names, h);
        install_built(c, h, &lib_id);
    }
    nb200_counts counts{};
    const int32_t rc = nb200_umi_counts(c, lib_id, R.key.size(), R.key.data(), R.off.data(), R.ids.data(), R.score.data(),
                                        umi_threshold, disable_thresholding, &counts);
    c->libs.pop_back();                                                     // the dictionary was only for this call
    if (rc != NB200_OK) return rc;
    write_counts_tsv(out_tsv, &counts, R.feature_names, R.cells);
    if (out3) {
        out3[0] = R.key.size(); out3[1] = counts.n_rows; out3[2] = counts.dropped_empty;
        if (disable_thresholding & NB200_UMI_CORRECT) out3[3] = c->umis_corrected;
    }
    API_END(c)
}

// Roofline denominator for the probe kernel: independent, uniformly random 32 B-sector gathers
// (one 256-bit load per thread per iteration, `loads_per_thread` in flight one after another)
// over a buffer of `bytes`.  Returns achieved GB/s (sector bytes) and loads/s.
namespace nb200 {
__global__ void __launch_bounds__(256)
random_gather_kernel(const uint4 *__restrict__ buf, uint64_t n_sectors, uint32_t iters, uint64_t seed, uint32_t *__restrict__ sink) {
    uint64_t x = seed + (uint64_t)(blockIdx.x * blockDim.x + threadIdx.x) * 0x9E3779B97F4A7C15ull;
    uint32_t acc = 0;
    for (uint32_t i = 0; i < iters; i += 4) {
        uint64_t idx[4];
#pragma unroll
        for (int u = 0; u < 4; u++) { x = dev_hash_kmer(x + 0x632BE59BD9B4E019ull); idx[u] = x % n_sectors; }
        uint4 lo[4], hi[4];
#pragma unroll
        for (int u = 0; u < 4; u++) ldg256(buf + 2 * idx[u], lo[u], hi[u]);
#pragma unroll
        for (int u = 0; u < 4; u++) acc += lo[u].x ^ hi[u].w;
    }
    if (acc == 0x12345678u) sink[0] = acc;      // keep the loads alive
}
}  // namespace nb200


// Roofline denominators for the Smith-Waterman kernel (SURVEY.md §8d): register-only loops at full occupancy.
//  dpx_peak_kernel: independent chains of the two DPX instructions sw_row issues, 2 : 1 like the kernel
//  (VIADDMNMX.S16x2.RELU, VIMNMX3.S16x2) -> DPX instructions per second.
//  sw_row_peak_kernel: the kernel's own row update (sw_row) on register-resident flags, no loads ->
//  cell updates per second the recurrence can reach on the integer pipe.
namespace nb200 {
__global__ void __launch_bounds__(256)
dpx_peak_kernel(uint32_t iters, uint32_t seed, uint32_t *__restrict__ sink) {
    uint32_t a[8], m[4];
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
#pragma unroll
    for (int j = 0; j < 8; j++) a[j] = (seed * (j + 3u) + t) & 0x0FFF0FFFu;
#pragma unroll
    for (int j = 0; j < 4; j++) m[j] = 0;
    const uint32_t g = seed | 0x00010001u, d = (seed >> 3) & 0x00FF00FFu;
    for (uint32_t i = 0; i < iters; i++) {
#pragma unroll
        for (int j = 0; j < 8; j++) a[j] = __viaddmax_s16x2_relu(a[j], g, d);
#pragma unroll
        for (int j = 0; j < 4; j++) m[j] = __vimax3_s16x2(m[j], a[2 * j], a[2 * j + 1]);
    }
    uint32_t acc = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) acc ^= m[j];
    if (acc == 0x12345677u) sink[0] = acc;
}

__global__ void __launch_bounds__(128)
sw_row_peak_kernel(uint32_t rows, uint32_t seed, uint32_t *__restrict__ sink) {
    uint32_t H[kNB];
#pragma unroll
    for (int b = 0; b < kNB; b++) H[b] = 0;
    uint32_t best = 0;
    uint32_t x = seed + (blockIdx.x * blockDim.x + threadIdx.x) * 0x9E3779B9u;
    for (uint32_t i = 0; i < rows; i++) {
        x = x * 1664525u + 1013904223u;                         // match flags of the row: one LCG step
        sw_row(H, x & 0x55555555u, (x >> 1) & 0x55555555u, (x >> 7) & 0x00010001u, best);
    }
    if (best == 0x12345677u) sink[0] = best;
}
}  // namespace nb200

int32_t nb200_bench_dpx_peak(nb200_ctx *c, uint32_t iters, double *dpx_ginst_per_s, double *row_gcups) {
    API_BEGIN(c)
    if (!dpx_ginst_per_s || !row_gcups || iters < 16) throw std::runtime_error("bad arguments");
    DevBuf sink;
    sink.ensure(64);
    Event e0, e1;
    CK(cudaEventCreate(&e0.h)); CK(cudaEventCreate(&e1.h));
    const unsigned b_dpx = (unsigned)c->sm_count * 8, b_row = (unsigned)c->sm_count * 16;
    auto time_best = [&](auto launch) {
        launch(16u);                                            // warm-up
        float best = 1e30f;
        for (int rep = 0; rep < 3; rep++) {
            CK(cudaEventRecord(e0, c->s_compute));
            launch(iters);
            CK(cudaEventRecord(e1, c->s_compute));
            CK(cudaStreamSynchronize(c->s_compute));
            float ms = 0;
            CK(cudaEventElapsedTime(&ms, e0, e1));
            best = std::min(best, ms);
        }
        return (double)best * 1e-3;
    };
    const double s_dpx = time_best([&](uint32_t it) { dpx_peak_kernel<<<b_dpx, 256, 0, c->s_compute>>>(it, 12345u + it, sink.as<uint32_t>()); });
    const double s_row = time_best([&](uint32_t it) { sw_row_peak_kernel<<<b_row, 128, 0, c->s_compute>>>(it, 999u + it, sink.as<uint32_t>()); });
    CK(cudaGetLastError());
    *dpx_ginst_per_s = (double)b_dpx * 256.0 * iters * 12.0 / s_dpx / 1e9;         // thread-level DPX instructions (s16x2 each)
    *row_gcups = (double)b_row * 128.0 * iters * (2.0 * kNB) / s_row / 1e9;         // two alignments per thread
    API_END(c)
}

// ---- fastq-to-bam -------------------------------------------------------------------------------
int32_t nb200_load_whitelist_mem(nb200_ctx *c, const char *entries, uint64_t n, int32_t cb_len, int32_t *wl_id) {
    API_BEGIN(c)
    if ((!entries && n) || !wl_id || cb_len < 1) throw std::runtime_error("bad arguments");
    std::vector<std::string> e;
    e.reserve(n);
    for (uint64_t i = 0; i < n; i++) e.emplace_back(entries + i * (size_t)cb_len, (size_t)cb_len);
    c->wls.push_back(build_whitelist(c, std::move(e), cb_len));
    *wl_id = (int32_t)c->wls.size() - 1;
    API_END(c)
}

int32_t nb200_load_whitelist(nb200_ctx *c, const char *path, int32_t cb_len, int32_t *wl_id) {
    API_BEGIN(c)
    if (!path || !wl_id) throw std::runtime_error("bad arguments");
    std::vector<std::string> e;
    read_whitelist_lines(path, e);
    c->wls.push_back(build_whitelist(c, std::move(e), cb_len));
    *wl_id = (int32_t)c->wls.size() - 1;
    API_END(c)
}

int32_t nb200_whitelist_info(const nb200_ctx *cc, int32_t wl_id, int64_t *n_entries, int64_t *n_unique, int64_t *table_bytes,
                             int32_t *cb_len) {
    nb200_ctx *c = const_cast<nb200_ctx *>(cc);
    API_BEGIN(c)
    const DevWhitelist &W = get_wl(c, wl_id);
    if (n_entries) *n_entries = (int64_t)W.entries.size();
    if (n_unique) *n_unique = (int64_t)W.n_unique;
    if (table_bytes) *table_bytes = (int64_t)(W.n_slots * sizeof(WlSlot));
    if (cb_len) *cb_len = W.cb_len;
    API_END(c)
}

const char *nb200_whitelist_entry(const nb200_ctx *c, int32_t wl_id, uint32_t idx) {
    if (!c || wl_id < 0 || wl_id >= (int32_t)c->wls.size() || idx >= c->wls[wl_id]->entries.size()) return nullptr;
    return c->wls[wl_id]->entries[idx].c_str();
}

int32_t nb200_cb_upload(nb200_ctx *c, int32_t cb_len, const char *cb, const uint8_t *qual, const uint8_t *eligible, uint64_t n) {
    API_BEGIN(c)
    if (cb_len < 1 || cb_len > kCbMaxLen || (n && (!cb || !qual))) throw std::runtime_error("bad arguments");
    cb_upload(c, cb_len, cb, qual, eligible, n, nullptr);
    CK(cudaStreamSynchronize(c->s_compute));
    API_END(c)
}

int32_t nb200_correct_barcodes_resident(nb200_ctx *c, int32_t wl_id, int32_t *out_idx, uint8_t *out_status, nb200_cb_stats *stats) {
    API_BEGIN(c)
    if (stats) memset(stats, 0, sizeof *stats);
    cb_run(c, get_wl(c, wl_id), stats);
    cb_fetch(c, out_idx, out_status, stats);
    if (stats) stats->total_ms = stats->kernel_ms;
    c->ev_pool.clear();
    API_END(c)
}

int32_t nb200_correct_barcodes(nb200_ctx *c, int32_t wl_id, const char *cb, const uint8_t *qual, const uint8_t *eligible,
                               uint64_t n, int32_t *out_idx, uint8_t *out_status, nb200_cb_stats *stats) {
    API_BEGIN(c)
    if (n && (!cb || !qual || !out_idx || !out_status)) throw std::runtime_error("bad arguments");
    DevWhitelist &W = get_wl(c, wl_id);
    if (stats) memset(stats, 0, sizeof *stats);
    cudaEvent_t e0 = new_event(c), e1 = new_event(c);
    CK(cudaEventRecord(e0, c->s_compute));
    cb_upload(c, W.cb_len, cb, qual, eligible, n, stats);
    cb_run(c, W, stats);
    cb_fetch(c, out_idx, out_status, stats);
    CK(cudaEventRecord(e1, c->s_compute));
    CK(cudaEventSynchronize(e1));
    if (stats) CK(cudaEventElapsedTime(&stats->total_ms, e0, e1));
    c->ev_pool.clear();
    API_END(c)
}

int32_t nb200_fastq_to_bam(nb200_ctx *c, const char *r1_fastq, const char *r2_fastq, const char *whitelist_path,
                           const char *output_bam, int32_t cb_len, int32_t umi_len, nb200_cb_stats *stats) {
    API_BEGIN(c)
    if (!r1_fastq || !r2_fastq || !whitelist_path || !output_bam || cb_len < 1 || umi_len < 0) throw std::runtime_error("bad arguments");
    nb200_cb_stats st{};
    std::vector<std::string> lines;
    read_whitelist_lines(whitelist_path, lines);
    std::unique_ptr<DevWhitelist> W = build_whitelist(c, std::move(lines), cb_len);
    FastqQ A, B;
    {
        std::string err;
        std::thread t([&] { try { load_fastq_qual(r2_fastq, B); } catch (const std::exception &e) { err = e.what(); } });
        try { load_fastq_qual(r1_fastq, A); } catch (...) { t.join(); throw; }
        t.join();
        if (!err.empty()) throw IoError(err);
    }
    const size_t n = std::min(A.recs.size(), B.recs.size());
    std::vector<uint8_t> cb(n * (size_t)cb_len + 16), qual(n * (size_t)cb_len + 16), elig(n + 16);
    slice_barcodes(A, B, cb_len, umi_len, c->host_threads, cb.data(), qual.data(), elig.data(), st);
    std::vector<int32_t> idx(n + 1);
    std::vector<uint8_t> status(n + 1);
    nb200_cb_stats dev{};
    cudaEvent_t e0 = new_event(c), e1 = new_event(c);
    CK(cudaEventRecord(e0, c->s_compute));
    cb_upload(c, cb_len, (const char *)cb.data(), qual.data(), elig.data(), n, &dev);
    cb_run(c, *W, &dev);
    cb_fetch(c, idx.data(), status.data(), &dev);
    CK(cudaEventRecord(e1, c->s_compute));
    CK(cudaEventSynchronize(e1));
    CK(cudaEventElapsedTime(&dev.total_ms, e0, e1));
    c->ev_pool.clear();
    dev.total_pairs = st.total_pairs; dev.name_mismatch = st.name_mismatch; dev.too_short = st.too_short;
    dev.no_remaining_seq = st.no_remaining_seq;
    write_10x_bam(output_bam, A, B, cb_len, umi_len, idx.data(), status.data(), W->entries, c->host_threads, dev);
    c->cb_resident = false;
    if (stats) *stats = dev;
    API_END(c)
}

int32_t nb200_bench_random_access(nb200_ctx *c, uint64_t bytes, uint32_t iters, double *gbytes_per_s, double *gloads_per_s) {
    API_BEGIN(c)
    if (bytes < (1u << 20) || !gbytes_per_s) throw std::runtime_error("bad arguments");
    DevBuf buf, sink;
    buf.ensure(bytes); sink.ensure(64);
    CK(cudaMemsetAsync(buf.p, 1, bytes, c->s_compute));
    const uint64_t n_sectors = bytes / 32;
    const unsigned blocks = (unsigned)c->sm_count * 16;
    iters = (iters + 3) & ~3u;
    Event e0, e1;
    CK(cudaEventCreate(&e0.h)); CK(cudaEventCreate(&e1.h));
    random_gather_kernel<<<blocks, 256, 0, c->s_compute>>>(buf.as<uint4>(), n_sectors, 64, 1, sink.as<uint32_t>());   // warm-up
    float best = 1e30f;
    for (int rep = 0; rep < 3; rep++) {
        CK(cudaEventRecord(e0, c->s_compute));
        random_gather_kernel<<<blocks, 256, 0, c->s_compute>>>(buf.as<uint4>(), n_sectors, iters, 17 + rep, sink.as<uint32_t>());
        CK(cudaEventRecord(e1, c->s_compute));
        CK(cudaStreamSynchronize(c->s_compute));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        best = std::min(best, ms);
    }
    const double loads = (double)blocks * 256.0 * iters;
    *gbytes_per_s = loads * 32.0 / (best * 1e-3) / 1e9;
    if (gloads_per_s) *gloads_per_s = loads / (best * 1e-3) / 1e9;
    API_END(c)
}

int32_t nb200_set_overlap(nb200_ctx *c, int32_t on) {
    if (!c) return NB200_EINVAL;
    c->overlap = on != 0;
    return NB200_OK;
}

int32_t nb200_set_defer_fetch(nb200_ctx *c, int32_t on) {
    if (!c) return NB200_EINVAL;
    c->defer_fetch = on ? 1 : 0;
    return NB200_OK;
}

// the four D2H copies of a deferred table, on the second copy stream (the device table is complete: nb200_align* returned)
static void start_table_fetch(nb200_ctx *c) {
    const uint64_t n_out = c->dev_rows, n_ids = c->dev_ids;
    ensure_host_table(c, n_out, n_ids);
    c->h_off.p[0] = 0;
    if (!c->fetch_pending || !n_out || c->fetch_started) return;
    cudaStream_t s = c->s_copy[1];
    CK(cudaMemcpyAsync(c->h_cell.p, c->o_cell_d.p, (size_t)n_out * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(c->h_count.p, c->o_count_d.p, (size_t)n_out * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(c->h_off.p, c->o_off_d.p, (size_t)(n_out + 1) * 4, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(c->h_ids.p, c->o_ids_d.p, (size_t)n_ids * 4, cudaMemcpyDeviceToHost, s));
    c->fetch_started = true;
}

int32_t nb200_fetch_counts_start(nb200_ctx *c) {
    API_BEGIN(c)
    start_table_fetch(c);
    API_END(c)
}

int32_t nb200_fetch_counts(nb200_ctx *c, nb200_counts *counts) {
    API_BEGIN(c)
    if (!counts) throw std::runtime_error("counts is null");
    const uint64_t n_out = c->dev_rows, n_ids = c->dev_ids;
    start_table_fetch(c);
    if (c->fetch_pending && n_out) {
        CK(cudaStreamSynchronize(c->s_copy[1]));
        c->fetch_started = false;
        if (c->h_off.p[n_out] != n_ids) throw std::runtime_error("internal: id count of the table disagrees with its offsets");
        c->timing.d2h_bytes += n_out * 12 + 4 + n_ids * 4;
        c->fetch_pending = false;
    }
    counts->n_rows = n_out;
    counts->cell = c->h_cell.p; counts->count = c->h_count.p; counts->feat_off = c->h_off.p; counts->feat_ids = c->h_ids.p;
    API_END(c)
}

int32_t nb200_set_stats(nb200_ctx *c, int32_t on) {
    if (!c) return NB200_EINVAL;
    c->stats = on != 0;
    return NB200_OK;
}

int32_t nb200_last_timing(const nb200_ctx *c, nb200_timing *out) {
    if (!c || !out) return NB200_EINVAL;
    *out = c->timing;
    return NB200_OK;
}

}  // extern "C"
