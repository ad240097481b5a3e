// sm_100a kernels of the 10x cell-barcode correction (SURVEY.md §8a A5, §8f rank 2).
// Semantics: DESIGN.md §2.8; bit-exact against oracle/cb_oracle.c, which is pinned on outputs of
// the reference's own functions (nimble/fastq_barcode_processor.py:17-36, :73-128).
//
// The reference materialises every 1-substitution variant of every whitelist entry in a Python
// dict (80 variants per 16-mer: ~0.5 G strings for a 6.8 M-entry 10x whitelist).  Here the
// whitelist is an open-addressing hash set in HBM (16 B slots) and the variants are enumerated
// from the READ side: one probe for the exact match (thread per read, streaming), and for the few
// reads that miss, 4 x cb_len variant probes spread over the lanes of a warp.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/nimble_b200.h"

namespace nb200 {

// Base codes in ASCII order (A < C < G < N < T), 3 bits each, position 0 in the most significant
// group: integer order of two keys == string order of the barcodes (the SPEC's tie order).
constexpr uint64_t kCbEmpty = ~0ull;          // code 7 never occurs: also marks "has a non-ACGTN base"
constexpr int kCbMaxLen = 21;

struct __align__(16) WlSlot {
    uint64_t key;
    uint32_t idx;     // index of the entry in the caller's whitelist (first occurrence)
    uint32_t pad;
};

struct WlDev {
    const WlSlot *table;
    uint64_t mask;
    int32_t cb_len;
};

struct CbCounters {
    unsigned long long n_miss, n_inval, perfect, corrected, none, n_multi, probes, pad;
};

__host__ __device__ __forceinline__ uint64_t cb_hash(uint64_t x) {
    x ^= x >> 29;
    x *= 0xD6E8FEB86659FD93ull;
    x ^= x >> 32;
    return x;
}

// 'A' 'C' 'G' 'N' 'T' -> 0..4, anything else -> 7.  (c >> 1) & 15 separates the five letters; the
// second table checks that the byte really is that letter.
__host__ __device__ __forceinline__ uint32_t cb_code(uint32_t c) {
    constexpr uint64_t kNib = 0x7777747737772710ull;                             // nibble[0]=0 [1]=1 [3]=2 [7]=3 [10]=4, else 7
    constexpr uint64_t kExp = 0x000000544E474341ull;                             // "ACGNT"
    const uint32_t code = (uint32_t)(kNib >> (4 * ((c >> 1) & 15))) & 7u;
    const uint32_t expect = (uint32_t)(kExp >> (8 * (code & 7u))) & 0xFFu;
    return (expect == c) ? code : 7u;
}

__device__ __forceinline__ int32_t wl_find(const WlDev &W, uint64_t key, uint32_t &probes) {
    uint64_t s = cb_hash(key) & W.mask;
    for (;;) {
        const uint4 v = __ldg(reinterpret_cast<const uint4 *>(W.table + s));
        probes++;
        const uint64_t k = ((uint64_t)v.y << 32) | v.x;
        if (k == key) return (int32_t)v.z;
        if (k == kCbEmpty) return -1;
        s = (s + 1) & W.mask;
    }
}

// Phase 1: thread per read.  Encode, exact lookup; misses go to miss_list (any order), reads
// with a base outside ACGTN-alphabet get NONE right away (no variant of a whitelist entry can
// contain such a byte) and are listed for the host's cache-size statistic.
__global__ void __launch_bounds__(256)
cb_exact_kernel(WlDev W, const uint8_t *__restrict__ cb, const uint8_t *__restrict__ eligible, uint64_t n,
                uint64_t *__restrict__ keys, int32_t *__restrict__ out_idx, uint8_t *__restrict__ out_status,
                uint32_t *__restrict__ miss_list, uint32_t *__restrict__ inval_list, uint32_t inval_cap,
                uint8_t *__restrict__ hit_flag, CbCounters *__restrict__ ctr) {
    __shared__ unsigned s_cnt[8], s_perfect, s_probes;
    __shared__ unsigned long long s_base;
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    if (threadIdx.x == 0) { s_perfect = 0; s_probes = 0; }
    const int L = W.cb_len;
    bool live = i < n;
    bool elig = live && (!eligible || eligible[i]);
    uint64_t key = 0;
    bool ok = true;
    if (elig) {
        if (L == 16) {
            const uint4 v = *reinterpret_cast<const uint4 *>(cb + i * 16);
            const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int j = 0; j < 16; j++) {
                const uint32_t c = cb_code((w[j >> 2] >> (8 * (j & 3))) & 0xFFu);
                ok &= c != 7u;
                key = (key << 3) | c;
            }
        } else {
            const uint8_t *p = cb + i * (uint64_t)L;
            for (int j = 0; j < L; j++) {
                const uint32_t c = cb_code(p[j]);
                ok &= c != 7u;
                key = (key << 3) | c;
            }
        }
    }
    uint32_t probes = 0;
    int32_t idx = -1;
    uint8_t status = NB200_CB_SKIPPED;
    if (elig) {
        if (!ok) { key = kCbEmpty; status = NB200_CB_NONE; }
        else {
            idx = wl_find(W, key, probes);
            status = idx >= 0 ? NB200_CB_PERFECT : NB200_CB_NONE;      // misses are revisited by phase 2
        }
    }
    if (live) {
        keys[i] = elig ? key : kCbEmpty;
        out_idx[i] = idx;
        out_status[i] = status;
    }
    if (hit_flag && idx >= 0) hit_flag[idx] = 1;       // distinct perfect barcodes = distinct entries hit
    // block-aggregated append of the misses and counters: one global atomic per block, not per warp
    // (a quarter of a million same-address atomics was 90 % of this kernel's time)
    const bool miss = elig && ok && idx < 0;
    const unsigned mb = __ballot_sync(0xFFFFFFFFu, miss);
    const unsigned pb = __ballot_sync(0xFFFFFFFFu, elig && idx >= 0);
    const uint32_t pr = __reduce_add_sync(0xFFFFFFFFu, probes);
    if (lane == 0) s_cnt[wib] = __popc(mb);
    __syncthreads();
    if (lane == 0) {
        if (pb) atomicAdd(&s_perfect, (unsigned)__popc(pb));
        if (pr) atomicAdd(&s_probes, pr);
    }
    if (threadIdx.x == 0) {
        unsigned tot = 0;
#pragma unroll
        for (int w = 0; w < 8; w++) { const unsigned c = s_cnt[w]; s_cnt[w] = tot; tot += c; }
        s_base = tot ? atomicAdd(&ctr->n_miss, (unsigned long long)tot) : 0ull;
    }
    __syncthreads();
    if (miss) miss_list[s_base + s_cnt[wib] + __popc(mb & ((1u << lane) - 1))] = (uint32_t)i;
    if (threadIdx.x == 0) {
        if (s_perfect) atomicAdd(&ctr->perfect, (unsigned long long)s_perfect);
        if (s_probes) atomicAdd(&ctr->probes, (unsigned long long)s_probes);
    }
    const bool inval = elig && !ok;                    // rare: warp-level append is fine
    const unsigned ib = __ballot_sync(0xFFFFFFFFu, inval);
    if (ib) {
        unsigned long long base = 0;
        if (lane == __ffs(ib) - 1) {
            base = atomicAdd(&ctr->n_inval, (unsigned long long)__popc(ib));
            atomicAdd(&ctr->none, (unsigned long long)__popc(ib));
        }
        base = __shfl_sync(0xFFFFFFFFu, base, __ffs(ib) - 1);
        const unsigned long long at = base + __popc(ib & ((1u << lane) - 1));
        if (inval && at < inval_cap) inval_list[at] = (uint32_t)i;
    }
}

// Phase 2: warp per missed read, persistent grid (the miss count stays on the device).
// Lane t handles variant (position t >> 2, t & 3-th other base); candidates are ranked by
// (quality at the differing position, candidate string) and the smallest wins.
__global__ void __launch_bounds__(128)
cb_hamming_kernel(WlDev W, const uint8_t *__restrict__ qual, const uint64_t *__restrict__ keys,
                  const uint32_t *__restrict__ miss_list, int32_t *__restrict__ out_idx, uint8_t *__restrict__ out_status,
                  uint8_t *__restrict__ multi_flag, CbCounters *__restrict__ ctr) {
    const int lane = threadIdx.x & 31;
    const uint32_t wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    const uint32_t n_miss = (uint32_t)ctr->n_miss;
    const int L = W.cb_len;
    uint32_t probes = 0, n_corr = 0, n_none = 0, n_multi = 0;
    for (uint32_t m = wid; m < n_miss; m += warps) {
        const uint32_t i = miss_list[m];
        const uint64_t key = keys[i];
        uint32_t best_q = 0xFFFFFFFFu, cnt = 0;
        uint64_t best_key = kCbEmpty;
        int32_t best_idx = -1;
        // two variants per lane and trip: both first probes are in flight before either is inspected
        for (int t0 = lane; t0 < 4 * L; t0 += 64) {
            uint64_t vkey[2], slot[2];
            uint4 v[2];
            int pos[2];
            bool live[2];
#pragma unroll
            for (int u = 0; u < 2; u++) {
                const int t = t0 + 32 * u;
                live[u] = t < 4 * L;
                pos[u] = live[u] ? (t >> 2) : 0;
                const int a = t & 3, sh = 3 * (L - 1 - pos[u]);
                const uint32_t cur = (uint32_t)(key >> sh) & 7u;
                const uint32_t sym = (uint32_t)a + ((uint32_t)a >= cur ? 1u : 0u);
                vkey[u] = key ^ ((uint64_t)(cur ^ sym) << sh);
                slot[u] = cb_hash(vkey[u]) & W.mask;
                if (live[u]) { v[u] = __ldg(reinterpret_cast<const uint4 *>(W.table + slot[u])); probes++; }
            }
#pragma unroll
            for (int u = 0; u < 2; u++) {
                if (!live[u]) continue;
                int32_t idx = -1;
                for (;;) {
                    const uint64_t k = ((uint64_t)v[u].y << 32) | v[u].x;
                    if (k == vkey[u]) { idx = (int32_t)v[u].z; break; }
                    if (k == kCbEmpty) break;
                    slot[u] = (slot[u] + 1) & W.mask;
                    v[u] = __ldg(reinterpret_cast<const uint4 *>(W.table + slot[u]));
                    probes++;
                }
                if (idx >= 0) {
                    cnt++;
                    const uint32_t q = qual[(uint64_t)i * L + pos[u]];
                    if (q < best_q || (q == best_q && vkey[u] < best_key)) { best_q = q; best_key = vkey[u]; best_idx = idx; }
                }
            }
        }
        const uint32_t total = __reduce_add_sync(0xFFFFFFFFu, cnt);
        if (total == 0) {
            if (lane == 0) n_none++;          // status is already NONE, idx -1
            continue;
        }
        const uint32_t mq = __reduce_min_sync(0xFFFFFFFFu, best_q);
        const uint64_t k = best_q == mq ? best_key : kCbEmpty;
        const uint32_t hi = __reduce_min_sync(0xFFFFFFFFu, (uint32_t)(k >> 32));
        const uint32_t lo = __reduce_min_sync(0xFFFFFFFFu, (uint32_t)(k >> 32) == hi ? (uint32_t)k : 0xFFFFFFFFu);
        const unsigned own = __ballot_sync(0xFFFFFFFFu, k == (((uint64_t)hi << 32) | lo));
        const int32_t idx = __shfl_sync(0xFFFFFFFFu, best_idx, __ffs(own) - 1);
        if (lane == 0) {
            out_idx[i] = idx;
            out_status[i] = NB200_CB_CORRECTED;
            n_corr++;
            if (total > 1) { multi_flag[i] = 1; n_multi++; }
        }
    }
    probes = __reduce_add_sync(0xFFFFFFFFu, probes);
    if (lane == 0) {
        if (n_corr) atomicAdd(&ctr->corrected, (unsigned long long)n_corr);
        if (n_none) atomicAdd(&ctr->none, (unsigned long long)n_none);
        if (n_multi) atomicAdd(&ctr->n_multi, (unsigned long long)n_multi);
        if (probes) atomicAdd(&ctr->probes, (unsigned long long)probes);
    }
}

// Phase 3 (the reference's correction_cache): among reads with SEVERAL candidates the first read
// in file order decides for every later read with the same raw barcode.  multi reads arrive sorted
// by (raw key, read index); head[t] = position of the first element of t's run.
__global__ void cb_gather_keys_kernel(const uint32_t *__restrict__ list, const uint64_t *__restrict__ keys, uint32_t m,
                                      uint64_t *__restrict__ out) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < m) out[t] = keys[list[t]];
}
__global__ void cb_run_heads_kernel(const uint64_t *__restrict__ sorted_keys, uint32_t m, uint32_t *__restrict__ head) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < m) head[t] = (t == 0 || sorted_keys[t] != sorted_keys[t - 1]) ? t : 0u;
}
__global__ void cb_propagate_kernel(const uint32_t *__restrict__ sorted_idx, const uint32_t *__restrict__ head, uint32_t m,
                                    int32_t *__restrict__ out_idx) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= m) return;
    const uint32_t h = head[t];
    if (h != t) out_idx[sorted_idx[t]] = out_idx[sorted_idx[h]];      // heads are never written: no race
}

// ---- fastq-to-counts (nb200_fastq_to_counts): one slab at a time, the cache rule over the whole call ----------------
// Per read of a slab: key = cell << 32 | umi.  On entry key holds the host's flags << 32 | umi (umi 0xFFFFFFFF for a
// pandas NA UMI; flags: slab_api.hpp kTenx*, a pair the two-step route refuses once it is written).  The flags of a read
// whose barcode is corrected (= written by fastq-to-bam) are or-ed into ctr->pad, which makes the host fail the call.
// cell = whitelist line for exact matches and single-candidate corrections (every read with that raw barcode gets the
// same answer).  A read with several candidates gets a provisional cell, bit 31 | its entry in the context's log, and is
// logged with its raw barcode, its file order and its own choice: lane_cb_resolve lets the first logged read of a raw
// barcode in file order decide for all of them.  Logged whatever its UMI: an uncounted read can still be the first.
__global__ void __launch_bounds__(256)
cb_key_kernel(uint32_t n, const uint8_t *__restrict__ status, const int32_t *__restrict__ idx, const uint8_t *__restrict__ multi,
              const uint64_t *__restrict__ raw, uint64_t order0, uint64_t *__restrict__ key, unsigned long long *__restrict__ log_n,
              uint64_t *__restrict__ log_key, uint64_t *__restrict__ log_order, int32_t *__restrict__ log_choice,
              CbCounters *__restrict__ ctr) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint8_t st = status[i];
    uint64_t k = NB200_NO_BARCODE;
    if (st == NB200_CB_PERFECT || st == NB200_CB_CORRECTED) {
        uint32_t cell = (uint32_t)idx[i];
        if (multi[i]) {
            const unsigned long long e = atomicAdd(log_n, 1ull);      // (rare: a few per cent of the reads at most)
            log_key[e] = raw[i];
            log_order[e] = order0 + i;
            log_choice[e] = idx[i];
            cell = 0x80000000u | (uint32_t)e;                         // (lane_cb_resolve refuses logs of 2^31 entries)
        }
        const uint64_t u = key[i];
        if ((uint32_t)u != 0xFFFFFFFFu) k = ((uint64_t)cell << 32) | (u & 0xFFFFFFFFull);
        if (u >> 32) atomicOr(&ctr->pad, (unsigned long long)(u >> 32));     // (rare)
    }
    key[i] = k;
}

// Gathered rows -> cell = rank of its whitelist line in byte order.  A provisional cell goes through decision[] first:
// rows [run_row[r], run_row[r + 1]) came from the log whose entries start at run_base[r] there.  A line that is a pandas
// NA token has rank ~0u: the row becomes NB200_NO_BARCODE (the UMI stage skips it) and is counted in *dropped.
__global__ void __launch_bounds__(256)
cb_remap_kernel(uint64_t n, uint64_t *__restrict__ key, const uint32_t *__restrict__ rank, const int32_t *__restrict__ decision,
                const uint64_t *__restrict__ run_row, const uint64_t *__restrict__ run_base, uint32_t n_runs,
                unsigned long long *__restrict__ dropped) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    bool drop = false;
    if (i < n) {
        const uint64_t k = key[i];
        uint32_t cell = (uint32_t)(k >> 32);
        if (cell & 0x80000000u) {
            uint32_t lo = 0, hi = n_runs;                              // last run with run_row[r] <= i
            while (hi - lo > 1) { const uint32_t m = (lo + hi) >> 1; if (run_row[m] <= i) lo = m; else hi = m; }
            cell = (uint32_t)decision[run_base[lo] + (cell & 0x7FFFFFFFu)];
        }
        const uint32_t r = rank[cell];
        drop = r == 0xFFFFFFFFu;
        key[i] = drop ? NB200_NO_BARCODE : (((uint64_t)r << 32) | (k & 0xFFFFFFFFull));
    }
    const unsigned b = __ballot_sync(0xFFFFFFFFu, drop);
    if ((threadIdx.x & 31) == 0 && b) atomicAdd(dropped, (unsigned long long)__popc(b));
}

__global__ void cb_count_flags_kernel(const uint8_t *__restrict__ flag, uint64_t n, unsigned long long *__restrict__ out) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned b = __ballot_sync(0xFFFFFFFFu, t < n && flag[t]);
    if ((threadIdx.x & 31) == 0 && b) atomicAdd(out, (unsigned long long)__popc(b));
}
__global__ void cb_count_distinct_kernel(const uint64_t *__restrict__ sorted_keys, uint64_t n, unsigned long long *__restrict__ out) {
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool h = t < n && sorted_keys[t] != kCbEmpty && (t == 0 || sorted_keys[t] != sorted_keys[t - 1]);
    const unsigned b = __ballot_sync(0xFFFFFFFFu, h);
    if ((threadIdx.x & 31) == 0 && b) atomicAdd(out, (unsigned long long)__popc(b));
}

}  // namespace nb200
