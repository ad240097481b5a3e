// sm_100a kernels of the read-assignment hot path (SURVEY.md §8a X3a, X3b, X3c, X4).
// Semantics: DESIGN.md §2 (SPEC); bit-exact against oracle/nimble_oracle.c.
//
// Equivalence classes and candidate sets are SPARSE bitsets over references: sorted
// (word index, 32 member bits) pairs.  A read's candidate set B starts as the narrowest class
// among its first hits and every further class is ANDed in with one warp-wide REDUX per word of B
// (lane = k-mer position), so the cost follows |B|'s width (2-3 words for allele families), not
// the library size.  Reads whose narrowest class is wider than kCap words take wide_kernel.
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/nimble_b200.h"
#include "kmer_hash.hpp"

namespace nb200 {

constexpr int kBand = 8;                 // SW half band
constexpr int kNB = 2 * kBand + 1;       // cells per row
constexpr int kVW = 64;                  // V = 64*score - edits
constexpr uint32_t kXP = 0xFF7FFF7Fu;    // packed s16x2 (-129,-129) mismatch
constexpr uint32_t kGP = 0xFF3FFF3Fu;    // packed s16x2 (-193,-193) gap
constexpr uint32_t kMatchDelta = 193;    // match - mismatch = 64 + 129
constexpr uint32_t kInvalid = 0xFFFFFFFFu;
constexpr int kCap = 32;                 // pairs per orientation kept in shared memory
constexpr int kScratchWords = 16 * kCap; // per warp: 4 lists + tmp + best (w and b arrays)
constexpr uint32_t kFull = 0xFFFFFFFFu;
constexpr int kProbeWarps = 2;           // warps per probe_kernel block (small blocks: occupancy follows the stragglers less)

struct LibDev {
    const uint4 *table;          // Entry[2 * n_buckets]: bucket = 2 x 16 B = one sector (library.hpp)
    uint32_t n_buckets;
    const uint4 *dual;           // DualRec[]: k-mers present on both strands
    const uint4 *class_rec;      // ClassRec[n_classes], 32 B each
    const uint32_t *ov_w, *ov_b, *ov_pre;
    const uint32_t *positions;
    const uint64_t *ref2bit;
    const uint32_t *refN;
    const uint32_t *ref_gstart;
    const uint32_t *ref_feature;
    uint32_t n_refs, n_features, n_words, narrow_cap;
    int32_t k, identity;
    uint64_t kmask, kbits;       // 2k low bits set / k low bits set
};

struct ReadsDev {
    const uint8_t *packed;
    const uint16_t *len;
    uint32_t stride, words;
};

struct __align__(16) RoRec {     // one mate in one orientation of a DEFERRED read
    uint32_t ncand;              // |B| (0 = empty intersection or no hit)
    uint32_t item_off;           // first SW item (kInvalid when none)
    uint16_t n_hits;
    uint16_t len;
    uint16_t na;                 // pairs parked in roB
    uint8_t full;                // every k-mer position hit -> no SW
    uint8_t pad;                 // 1: every candidate set of the read has at most 4 words (thread-per-read deferred call)
};

struct __align__(16) SwItem {
    uint32_t ro;                 // bits 0-21: deferred slot * n_ro + orientation; bits 22-30: read length
    uint32_t ref;                // candidate reference (kInvalid = padding)
    uint32_t gwin;               // global coordinate of band cell (row 0, b 0)
    uint32_t v;                  // out: best V
};

struct CallParams {
    int32_t score_threshold, score_filter, num_mismatches, discard_multiple_matches, intersect_level,
        discard_multi_hits, require_valid_pair, max_hits, strand_filter;
    // score_percent as a table: min_score[len] = smallest score s for which (double)s / (double)len < score_percent is
    // false (built on the host with that very expression, engine.cu), so the kernels need no FP64 division
    const uint16_t *min_score;
};

constexpr int kCtrSpread = 64;   // statistics counters are spread over 64 slots to avoid same-address REDs
struct Counters {
    // alloc = (deferred reads << 40) | SW items : one atomic hands out both cursors
    unsigned long long alloc, overflow, dropped_empty, max_nf, sw_pairs, sw_cells, items_max, deferred_total;
    unsigned long long n_wide, wide_total, n_swpairs, sw_dups, sw_items, n_slow, n_setup, n_warpdef;
    unsigned long long probes[kCtrSpread], probe_slots[kCtrSpread];
    unsigned long long n_probe_warp, probe_warp_total;   // reads probe_thread_kernel left to the warp form (batch / call)
};
constexpr unsigned long long kItemMask = (1ull << 40) - 1;
constexpr int kRoIdxBits = 22;               // a batch holds at most 2^22 read orientations (engine.cu: 2^21 reads x 2, 2^20 pairs x 4)
constexpr uint32_t kRoIdxMask = (1u << kRoIdxBits) - 1;

__device__ __forceinline__ uint64_t dev_hash_kmer(uint64_t x) {   // identical to hash_kmer (library.cpp)
    x ^= x >> 29;
    x *= 0xD6E8FEB86659FD93ull;
    x ^= x >> 32;
    return x;
}

__device__ __forceinline__ uint64_t dev_revcomp(uint64_t x, int k) {
    uint64_t r = __brevll(~x);
    r = ((r >> 1) & 0x5555555555555555ull) | ((r & 0x5555555555555555ull) << 1);
    return r >> (64 - 2 * k);
}

// one 32 B record = one L2 sector, fetched with a single 256-bit load that bypasses L1
__device__ __forceinline__ void ldg256(const uint4 *p, uint4 &lo, uint4 &hi) {
    asm volatile("ld.global.nc.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(lo.x), "=r"(lo.y), "=r"(lo.z), "=r"(lo.w), "=r"(hi.x), "=r"(hi.y), "=r"(hi.z), "=r"(hi.w)
                 : "l"(p));
}
__device__ __forceinline__ void ldg256_cached(const uint4 *p, uint4 &lo, uint4 &hi) {   // class records: reuse in L1
    asm volatile("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(lo.x), "=r"(lo.y), "=r"(lo.z), "=r"(lo.w), "=r"(hi.x), "=r"(hi.y), "=r"(hi.z), "=r"(hi.w)
                 : "l"(p));
}

__device__ __forceinline__ uint32_t warp_sum(uint32_t v) { return __reduce_add_sync(kFull, v); }
__device__ __forceinline__ uint32_t warp_max(uint32_t v) { return __reduce_max_sync(kFull, v); }
__device__ __forceinline__ uint32_t warp_excl_scan(uint32_t v, int lane, uint32_t &total) {
    uint32_t inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(kFull, inc, o);
        if (lane >= o) inc += t;
    }
    total = __shfl_sync(kFull, inc, 31);
    return inc - v;
}

enum { ST_NONE = 0, ST_PASS = 1, ST_NO_MATCH = 2, ST_EMPTY = 3, ST_SCORE = 4, ST_PERCENT = 5, ST_MULTI = 6 };
enum { RS_CALLED = 0, RS_NO_PASS = 1, RS_NOT_VALID_PAIR = 2, RS_FORCE_INTERSECT = 3, RS_SCORE_FILTER = 4,
       RS_MULTI_HITS = 5, RS_MAX_HITS = 6 };

// ---- class records (ClassRec, library.hpp) ----------------------------------------------------------
struct Rec {
    uint32_t n;                  // pairs (true count for the overflow form)
    uint32_t w[4], b[4];         // inline pairs (unused: w = 0xFFFF, b = 0); overflow: b[0] = offset
    bool inl;
};

__device__ __forceinline__ Rec unpack_rec(const uint4 lo, const uint4 hi) {   // lo: bits, hi: (w01, w23, meta, spare)
    Rec r;
    r.b[0] = lo.x; r.b[1] = lo.y; r.b[2] = lo.z; r.b[3] = lo.w;
    r.w[0] = hi.x & 0xFFFFu; r.w[1] = hi.x >> 16; r.w[2] = hi.y & 0xFFFFu; r.w[3] = hi.y >> 16;
    r.inl = (int32_t)hi.z >= 0;
    r.n = r.inl ? (hi.z & 0xFFu) : lo.y;
    return r;
}
__device__ __forceinline__ Rec empty_rec() {
    Rec r;
    r.n = 0; r.inl = true;
#pragma unroll
    for (int t = 0; t < 4; t++) { r.w[t] = 0xFFFFu; r.b[t] = 0; }
    return r;
}

__device__ __forceinline__ Rec load_rec(const LibDev &lib, uint32_t cls) {
    uint4 lo, hi;
    ldg256_cached(lib.class_rec + 2 * (size_t)cls, lo, hi);
    return unpack_rec(lo, hi);
}

// index of `word` in the overflow list, or -1
__device__ __forceinline__ int ov_find(const LibDev &lib, uint32_t off, uint32_t cnt, uint32_t word) {
    uint32_t lo = 0, hi = cnt;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (__ldg(lib.ov_w + off + mid) < word) lo = mid + 1; else hi = mid;
    }
    return (lo < cnt && __ldg(lib.ov_w + off + lo) == word) ? (int)lo : -1;
}

// member bits of the class at reference word `word`
__device__ __forceinline__ uint32_t rec_lookup(const LibDev &lib, const Rec &r, uint32_t word) {
    if (r.inl) {
        uint32_t v = 0;
#pragma unroll
        for (int i = 0; i < 4; i++) v |= (r.w[i] == word) ? r.b[i] : 0u;     // unused pairs match no word
        return v;
    }
    const int i = ov_find(lib, r.b[0], r.n, word);
    return i < 0 ? 0u : __ldg(lib.ov_b + r.b[0] + i);
}

// rank of reference `ref` among the class members (ref must be a member)
__device__ __forceinline__ uint32_t rec_rank(const LibDev &lib, const Rec &r, uint32_t ref) {
    const uint32_t word = ref >> 5, below = (1u << (ref & 31)) - 1;
    if (r.inl) {
        uint32_t rank = 0;
#pragma unroll
        for (int i = 0; i < 4; i++) {
            if (r.w[i] < word) rank += __popc(r.b[i]);                       // unused pairs: w = 0xFFFF > any word
            else if (r.w[i] == word) rank += __popc(r.b[i] & below);
        }
        return rank;
    }
    const int i = ov_find(lib, r.b[0], r.n, word);
    return __ldg(lib.ov_pre + r.b[0] + i) + __popc(__ldg(lib.ov_b + r.b[0] + i) & below);
}

// ---- sparse lists in scratch (shared memory for narrow reads, global for wide ones) -----------------
struct List {
    uint32_t *w, *b;
    int n;
};

__device__ __forceinline__ int list_find(const List &A, uint32_t word) {
    int lo = 0, hi = A.n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (A.w[mid] < word) lo = mid + 1; else hi = mid;
    }
    return (lo < A.n && A.w[lo] == word) ? lo : -1;
}
__device__ __forceinline__ uint32_t list_lookup(const List &A, uint32_t word) {
    const int i = list_find(A, word);
    return i < 0 ? 0u : A.b[i];
}
__device__ __forceinline__ uint32_t list_count(const List &A, int lane) {
    if (A.n <= 32) return warp_sum(lane < A.n ? (uint32_t)__popc(A.b[lane]) : 0u);
    uint32_t c = 0;
    for (int j = lane; j < A.n; j += 32) c += __popc(A.b[j]);
    return warp_sum(c);
}
__device__ __forceinline__ void list_copy(List &D, const List &A, int lane) {
    for (int j = lane; j < A.n; j += 32) { D.w[j] = A.w[j]; D.b[j] = A.b[j]; }
    D.n = A.n;
    __syncwarp();
}
// D = A & B on A's words; returns whether any bit survives
__device__ __forceinline__ bool list_intersect(List &D, const List &A, const List &B, int lane) {
    uint32_t any = 0;
    for (int j = lane; j < A.n; j += 32) {
        const uint32_t v = A.b[j] & list_lookup(B, A.w[j]);
        D.w[j] = A.w[j]; D.b[j] = v;
        any |= v;
    }
    D.n = A.n;
    __syncwarp();
    return __any_sync(kFull, any != 0);
}
// D = A | B (sorted merge; the lists are a handful of pairs, one lane does it)
__device__ __forceinline__ void list_union(List &D, const List &A, const List &B, int lane) {
    int n = 0;
    if (lane == 0) {
        int i = 0, j = 0;
        while (i < A.n || j < B.n) {
            if (j >= B.n || (i < A.n && A.w[i] < B.w[j])) { D.w[n] = A.w[i]; D.b[n] = A.b[i]; i++; }
            else if (i >= A.n || B.w[j] < A.w[i]) { D.w[n] = B.w[j]; D.b[n] = B.b[j]; j++; }
            else { D.w[n] = A.w[i]; D.b[n] = A.b[i] | B.b[j]; i++; j++; }
            n++;
        }
    }
    D.n = __shfl_sync(kFull, n, 0);
    __syncwarp();
}

// Everything the score/feature stage needs about one read (pair): 4 orientations.
struct ReadState {
    List cls[4];                // B' per orientation
    uint32_t nc[4], nh[4];
    int vbest[4];               // -1: no class (no hit / empty)
    int len[4];
    int n_sw;
};

// ---------------------------------------------------------------------------------------------
// X4: score / strand / pair filter + feature calling (DESIGN.md §2.5-2.6).  Warp-cooperative.
// T and Bst are scratch lists (capacity 2x an orientation list).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void call_read(const LibDev &lib, const CallParams &cp, bool paired, ReadState &S,
                                          List T, List Bst, int lane, nb200_read_result *res_out, int32_t *fout,
                                          uint16_t *nf_out, Counters *ctr) {
    int st[4], sc[4], ed[4];
#pragma unroll
    for (int o = 0; o < 4; o++) {
        st[o] = ST_NONE; sc[o] = 0; ed[o] = 0;
        if (!paired && o >= 2) continue;
        if (S.nh[o] == 0) { st[o] = ST_NO_MATCH; continue; }
        if (S.vbest[o] < 0) { st[o] = ST_EMPTY; continue; }
        sc[o] = (S.vbest[o] + kVW - 1) / kVW;
        ed[o] = sc[o] * kVW - S.vbest[o];
        if (sc[o] < cp.score_threshold) st[o] = ST_SCORE;
        else if (sc[o] < (int)cp.min_score[S.len[o]]) st[o] = ST_PERCENT;     // == (double)score / (double)len < score_percent
        else if (cp.discard_multiple_matches && S.nc[o] > 1) st[o] = ST_MULTI;
        else st[o] = ST_PASS;
    }
    int order[4], n_cfg = 0;
    const bool any_pass = st[0] == ST_PASS || st[1] == ST_PASS || st[2] == ST_PASS || st[3] == ST_PASS;
    switch (any_pass ? cp.strand_filter : -1) {
    case -1: break;            // no orientation passed: every configuration fails the same way (below)
    case NB200_FIVEPRIME: order[n_cfg++] = 0; break;
    case NB200_THREEPRIME: order[n_cfg++] = 1; break;
    case NB200_STRAND_NONE: order[n_cfg++] = 0; order[n_cfg++] = 1; if (paired) { order[n_cfg++] = 2; order[n_cfg++] = 3; } break;
    default: order[n_cfg++] = 0; order[n_cfg++] = 1; break;
    }
    // with no passing orientation every configuration fails at the same test (SPEC §2.6 order)
    int chosen = -1, chosen_max = 0;
    int first_fail = (!any_pass && paired && cp.require_valid_pair) ? RS_NOT_VALID_PAIR : RS_NO_PASS;
    uint32_t chosen_score = 0;
    List Tb = Bst;             // scratch copy target
    Bst.n = 0;
#pragma unroll
    for (int ci = 0; ci < 4; ci++) {
        if (ci >= n_cfg) continue;
        const int c = order[ci];
        const int ia = (c == 0 || c == 2) ? 0 : 1;            // F,FF: r1 fwd ; R,RR: r1 rc
        const int ib = (c == 0 || c == 3) ? 3 : 2;            // F,RR: r2 rc  ; R,FF: r2 fwd
        const int sa = ia == 0 ? sc[0] : sc[1], sbv = ib == 3 ? sc[3] : sc[2];
        const bool pa = (ia == 0 ? st[0] : st[1]) == ST_PASS, pb = paired && (ib == 3 ? st[3] : st[2]) == ST_PASS;
        const List A = ia == 0 ? S.cls[0] : S.cls[1];
        const List B = ib == 3 ? S.cls[3] : S.cls[2];
        int fail = -1, maxmate = 0;
        uint32_t s = 0;
        int src = 0;           // where the configuration's class lives: 0 = A, 1 = B, 2 = T (computed)
        if (!paired) {
            if (!pa) fail = RS_NO_PASS;
            else { s = (uint32_t)sa; maxmate = sa; src = 0; }
        } else if (cp.require_valid_pair && !(pa && pb)) fail = RS_NOT_VALID_PAIR;
        else if (!pa && !pb) fail = RS_NO_PASS;
        else if (pa && pb) {
            s = (uint32_t)(sa + sbv); maxmate = max(sa, sbv);
            if (cp.intersect_level == 0) { list_union(T, A, B, lane); src = 2; }
            else if (list_intersect(T, A, B, lane)) src = 2;
            else if (cp.intersect_level >= 2) fail = RS_FORCE_INTERSECT;
            else src = (sbv > sa) ? 1 : 0;
        } else {
            if (cp.intersect_level >= 2) fail = RS_FORCE_INTERSECT;
            else { src = pa ? 0 : 1; s = (uint32_t)(pa ? sa : sbv); maxmate = (int)s; }
        }
        if (fail >= 0) { if (ci == 0) first_fail = fail; continue; }
        if (chosen < 0 || s > chosen_score) {
            chosen = c; chosen_score = s; chosen_max = maxmate;
            if (src == 2) { list_copy(Tb, T, lane); Bst = Tb; }   // T is reused by the next configuration
            else Bst = src == 0 ? A : B;                           // orientation lists are read-only here
        }
    }
    int reason = first_fail, n_feat = 0;
    const int mh = cp.max_hits;
    if (chosen >= 0) {
        if (chosen_max < cp.score_filter) reason = RS_SCORE_FILTER;
        else if (lib.identity) {
            const int nf = (int)list_count(Bst, lane);
            if (cp.discard_multi_hits > 0 && nf > cp.discard_multi_hits) reason = RS_MULTI_HITS;
            else if (nf > mh) reason = RS_MAX_HITS;
            else {
                reason = RS_CALLED; n_feat = nf;
                uint32_t run = 0;
                for (int base = 0; base < Bst.n; base += 32) {
                    const int j = base + lane;
                    uint32_t bits = j < Bst.n ? Bst.b[j] : 0u, tot;
                    uint32_t ex = run + warp_excl_scan(__popc(bits), lane, tot);
                    while (bits) {
                        const int b = __ffs(bits) - 1;
                        bits &= bits - 1;
                        fout[ex++] = (int32_t)(Bst.w[j] * 32 + b);
                    }
                    run += tot;
                }
            }
        } else {
            // references are ordered by feature, so features of ascending members are non-decreasing:
            // a feature starts where it differs from the previous member's.  Pass 0 counts, pass 1 writes.
            for (int pass = 0; pass < 2; pass++) {
                uint32_t run = 0, total = 0;
                uint32_t prev_last = kInvalid;      // feature of the last member of earlier chunks
                for (int base = 0; base < Bst.n; base += 32) {
                    const int j = base + lane;
                    const uint32_t bits0 = j < Bst.n ? Bst.b[j] : 0u;
                    const uint32_t wbase = j < Bst.n ? Bst.w[j] * 32 : 0u;
                    const uint32_t mylast = bits0 ? __ldg(lib.ref_feature + wbase + (31 - __clz(bits0))) : kInvalid;
                    const unsigned ne = __ballot_sync(kFull, bits0 != 0);
                    const unsigned lower = ne & ((1u << lane) - 1);
                    uint32_t prev = __shfl_sync(kFull, mylast, lower ? 31 - __clz(lower) : 0);
                    if (!lower) prev = prev_last;
                    uint32_t cnt = 0, p2 = prev, bb = bits0;
                    while (bb) {
                        const int b = __ffs(bb) - 1;
                        bb &= bb - 1;
                        const uint32_t f = __ldg(lib.ref_feature + wbase + b);
                        if (f != p2) { cnt++; p2 = f; }
                    }
                    uint32_t tot;
                    uint32_t ex = run + warp_excl_scan(cnt, lane, tot);
                    if (pass == 1) {
                        p2 = prev; bb = bits0;
                        while (bb) {
                            const int b = __ffs(bb) - 1;
                            bb &= bb - 1;
                            const uint32_t f = __ldg(lib.ref_feature + wbase + b);
                            if (f != p2) { fout[ex++] = (int32_t)f; p2 = f; }
                        }
                    }
                    run += tot; total += tot;
                    if (ne) prev_last = __shfl_sync(kFull, mylast, 31 - __clz(ne));
                }
                if (pass == 0) {
                    const int nf = (int)total;
                    if (cp.discard_multi_hits > 0 && nf > cp.discard_multi_hits) { reason = RS_MULTI_HITS; break; }
                    if (nf > mh) { reason = RS_MAX_HITS; break; }
                    reason = RS_CALLED; n_feat = nf;
                }
            }
        }
    }
    __syncwarp();
    if (mh <= 32) { if (lane >= n_feat && lane < mh) fout[lane] = -1; }
    else for (int t = n_feat + lane; t < mh; t += 32) fout[t] = -1;
    if (lane == 0) {
        nb200_read_result res;
#pragma unroll
        for (int o = 0; o < 4; o++) {
            res.score[o] = (uint16_t)sc[o]; res.n_hits[o] = (uint16_t)S.nh[o];
            res.n_cand[o] = (uint16_t)(S.nc[o] > 65535u ? 65535u : S.nc[o]);
            res.edits[o] = (uint8_t)ed[o]; res.status[o] = (uint8_t)st[o];
        }
        res.reason = (uint8_t)reason; res.config = (uint8_t)(chosen < 0 ? 255 : chosen);
        res.n_feat = (uint8_t)n_feat; res.n_sw = (uint8_t)S.n_sw;
        res.pair_score = chosen < 0 ? 0u : chosen_score;
        *res_out = res;
        *nf_out = (uint16_t)n_feat;
    }
}

// ---------------------------------------------------------------------------------------------
// X3a + X3b for one mate.  Lane = k-mer position, 32 positions per round, rounds in a ROLLED loop (the probe
// kernel is bound by instruction issue and instruction fetch: the hot loop stays a few hundred instructions).
//
// Lookup (mirrors host_lookup in library.cpp, which the CPU suite checks for every library k-mer): k-mer and
// its reverse complement in 32-bit halves, canonical form, kmer_mix -> first bucket, ONE 256-bit load (two
// 16 B entries).  The second bucket is read only where the first carries the spill bit and does not hold the key,
// behind a warp vote, so most rounds never execute that path; same for entries of k-mers present on both
// strands (dual records).
//
// Intersection: B starts as the narrowest class among the first hits (at most 4 sparse words in the fast path,
// kept in registers); every lane ANDs the member bits of its own class into per-word accumulators, round after
// round, and ONE REDUX per word at the very end gives B.  Wider anchors and overflow-form classes take the
// generic path (lists in memory, one REDUX per word and round).
// Returns false when the read must take the wide path.
// ---------------------------------------------------------------------------------------------
constexpr uint32_t kDevSpill = 1u << 29, kDevRc = 1u << 30, kDevDual = 1u << 31, kDevIdMask = kDevSpill - 1;

struct RegB { uint32_t w01, w23, b0, b1, b2, b3; };    // a candidate set of at most 4 sparse words (word indices packed 16 + 16)
struct MateProbe {
    uint32_t nh[2];
    int seed_i[2];              // position of the seed k-mer in the ORIENTED read
    int L, P;
    int owner;                  // orientation whose candidate set came back in `reg` (-1: none); its list holds only n
    RegB reg;
};

// What the probe leaves per mate and orientation for the calling kernels: 32 B.
struct __align__(16) OriSum {
    uint16_t nh;                // index k-mers hit
    int16_t seed_i;             // position of the seed k-mer in the oriented read
    uint8_t na;                 // sparse words of the candidate set B
    uint8_t flags;              // kSumFull | kSumInMem | kSumWide
    uint16_t len;               // read length
    uint32_t w01, w23;          // word indices (na <= 4), 16 bits each
    uint32_t b[4];              // member bits
};
static_assert(sizeof(OriSum) == 32, "two 16-byte stores per orientation");
constexpr uint8_t kSumFull = 1;     // every k-mer position hit: no alignment needed
constexpr uint8_t kSumInMem = 2;    // B has more than 4 words: it lives in the batch's list area (roB), read-indexed
constexpr uint8_t kSumWide = 128;   // the read went to wide_kernel (flag on orientation 0 only)

__device__ __forceinline__ int read_length(const ReadsDev &R, uint64_t read) {   // never beyond the packed record
    return min((int)R.len[read], (int)R.words * 32);
}

// Class and position offset of the seed k-mer of an oriented read (the probe loop only keeps its position): one table
// lookup, same protocol as the loop (and as host_lookup in library.cpp), done by every lane alike.  Only reads that go
// to Smith-Waterman need it.
__device__ __forceinline__ void seed_lookup(const LibDev &lib, const ReadsDev &R, uint64_t read, int P, int o, int seed_i,
                                            uint32_t &cls, uint32_t &off) {
    const uint8_t *rec = R.packed + read * R.stride;
    const uint64_t *seq = reinterpret_cast<const uint64_t *>(rec);
    const int p = o ? P - 1 - seed_i : seed_i;                 // position in the read as sequenced
    const int w = p >> 5, sh = 2 * (p & 31);
    const uint64_t a = seq[w], b = (w + 1 < (int)R.words) ? seq[w + 1] : 0ull;
    const uint64_t x = (sh ? ((a >> sh) | (b << (64 - sh))) : a) & lib.kmask;
    const uint64_t y = dev_revcomp(x, lib.k);
    const uint64_t c = x < y ? x : y;
    const uint32_t c_lo = (uint32_t)c, c_hi = (uint32_t)(c >> 32);
    const uint32_t mix = kmer_mix(c_lo, c_hi), b1 = kmer_bucket1(mix, lib.n_buckets);
    uint4 e_lo, e_hi;
    ldg256(lib.table + 2 * (size_t)b1, e_lo, e_hi);
    bool m0 = e_lo.x == c_lo && e_lo.y == c_hi, m1 = e_hi.x == c_lo && e_hi.y == c_hi;
    if (!(m0 || m1)) {                                         // the seed is a hit: it must be in its second bucket
        ldg256(lib.table + 2 * (size_t)kmer_bucket2(mix, c_lo, b1, lib.n_buckets), e_lo, e_hi);
        m0 = e_lo.x == c_lo && e_lo.y == c_hi; m1 = e_hi.x == c_lo && e_hi.y == c_hi;
    }
    const uint32_t ecls = m0 ? e_lo.z : e_hi.z, eoff = m0 ? e_lo.w : e_hi.w;
    cls = ecls & kDevIdMask; off = eoff;
    if (ecls & kDevDual) {
        const uint4 d = __ldg(lib.dual + (ecls & kDevIdMask));
        const bool own = o ? (y <= x) : (x <= y);              // orientation o reads the canonical form itself
        cls = own ? d.x : d.z; off = own ? d.y : d.w;
    }
}

__device__ __forceinline__ uint32_t rec_lookup_overflow(const uint32_t *ov_w, const uint32_t *ov_b, uint32_t off, uint32_t cnt, uint32_t word) {
    uint32_t lo = 0, hi = cnt;
#pragma unroll 1
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (__ldg(ov_w + off + mid) < word) lo = mid + 1; else hi = mid;
    }
    return (lo < cnt && __ldg(ov_w + off + lo) == word) ? __ldg(ov_b + off + lo) : 0u;
}

// member bits of a class at `word`.  c_b: the four bit words; c_w: (w01, w23, meta, -) as loaded
__device__ __forceinline__ uint32_t rec_bits(const LibDev &lib, const uint4 c_b, const uint4 c_w, uint32_t word) {
    if ((int32_t)c_w.z >= 0) {
        uint32_t v = (c_w.x & 0xFFFFu) == word ? c_b.x : 0u;
        v = (c_w.x >> 16) == word ? c_b.y : v;      // word indices of a record are distinct: at most one matches
        v = (c_w.y & 0xFFFFu) == word ? c_b.z : v;
        v = (c_w.y >> 16) == word ? c_b.w : v;
        return v;
    }
    return rec_lookup_overflow(lib.ov_w, lib.ov_b, c_b.x, c_b.y, word);
}

// generic intersection step (B in memory: anchors wider than 4 words, or the second orientation of a read that
// hits on both strands): one REDUX per word of B and round.  Rare.
__device__ __forceinline__ bool intersect_generic(const LibDev &lib, uint32_t *lw, uint32_t *lb, int n, bool hit, uint4 c_b, uint4 c_w, int lane) {
    uint32_t alive = 0;
#pragma unroll 1
    for (int j = 0; j < n; j++) {
        const uint32_t v = hit ? rec_bits(lib, c_b, c_w, lw[j]) : kFull;
        const uint32_t nbits = lb[j] & __reduce_and_sync(kFull, v);
        __syncwarp();
        if (lane == (j & 31)) lb[j] = nbits;
        alive |= nbits;
    }
    __syncwarp();
    return alive != 0;
}
// anchor class -> list in memory (src lane holds the record)
__device__ __forceinline__ void anchor_to_list(const LibDev &lib, uint32_t *lw, uint32_t *lb, uint32_t nn, uint4 c_b, uint4 c_w, int src, int lane) {
    if (nn <= 4) {
        if (lane == src) {
            lw[0] = c_w.x & 0xFFFFu; lb[0] = c_b.x;
            if (nn > 1) { lw[1] = c_w.x >> 16; lb[1] = c_b.y; }
            if (nn > 2) { lw[2] = c_w.y & 0xFFFFu; lb[2] = c_b.z; }
            if (nn > 3) { lw[3] = c_w.y >> 16; lb[3] = c_b.w; }
        }
    } else {
        const uint32_t src_off = __shfl_sync(kFull, c_b.x, src);
#pragma unroll 1
        for (uint32_t t = lane; t < nn; t += 32) { lw[t] = __ldg(lib.ov_w + src_off + t); lb[t] = __ldg(lib.ov_b + src_off + t); }
    }
    __syncwarp();
}

// State of the orientation whose candidate set B lives in registers (the first orientation of the read that hits,
// when its anchor class has at most 4 words): B's packed word indices, the anchor's bits, the AND accumulators.
struct OwnerB {
    uint32_t w01, w23, b0, b1, b2, b3, a0, a1, a2, a3;
};

// one round of one orientation: anchor selection on the first hits, then B &= the classes hit in this round
// returns false when the read must take the wide path
__device__ __forceinline__ bool candidate_round(const LibDev &lib, const int o, const uint32_t cl, uint32_t cap, int lane, uint32_t *lw, uint32_t *lb,
                                                int &na, int &owner, bool &dead, OwnerB &B) {
    const bool hit = cl != kInvalid;
    uint4 c_b, c_w;
    ldg256_cached(lib.class_rec + 2 * (size_t)(hit ? cl : 0u), c_b, c_w);      // lanes without a hit read record 0 and ignore it
    const bool inl = (int32_t)c_w.z >= 0;
    if (na < 0) {
        // anchor = narrowest class among this round's hits; B can only shrink from it
        const uint32_t cn = inl ? (c_w.z & 0xFFu) : c_b.y;                      // pairs of the class
        const uint32_t m = __reduce_min_sync(kFull, hit ? ((min(cn, 0x3FFFFFFu) << 5) | (uint32_t)lane) : kInvalid);
        const int src = (int)(m & 31);
        const uint32_t nn = m >> 5;
        if (nn > cap) return false;
        na = (int)nn;
        if (nn <= 4 && owner < 0) {                 // an inline record by construction: B in registers
            owner = o;
            B.w01 = __shfl_sync(kFull, c_w.x, src); B.w23 = __shfl_sync(kFull, c_w.y, src);
            B.b0 = __shfl_sync(kFull, c_b.x, src); B.b1 = __shfl_sync(kFull, c_b.y, src);
            B.b2 = __shfl_sync(kFull, c_b.z, src); B.b3 = __shfl_sync(kFull, c_b.w, src);
        } else {
            anchor_to_list(lib, lw, lb, nn, c_b, c_w, src, lane);
        }
    }
    if (o == owner) {
        // Classes of an allele family mostly span the same reference words as B: then the AND is word by word.
        const bool same = !hit || (c_w.x == B.w01 && c_w.y == B.w23 && inl);
        if (__all_sync(kFull, same)) {
            if (hit) { B.a0 &= c_b.x; B.a1 &= c_b.y; B.a2 &= c_b.z; B.a3 &= c_b.w; }
        } else {
            // general: look B's words up in the lane's class (unused words of B: 0xFFFF, matched by unused words of the
            // class with zero bits; their accumulators are never read)
            if (hit && inl) {
                B.a0 &= rec_bits(lib, c_b, c_w, B.w01 & 0xFFFFu);
                B.a1 &= rec_bits(lib, c_b, c_w, B.w01 >> 16);
                B.a2 &= rec_bits(lib, c_b, c_w, B.w23 & 0xFFFFu);
                B.a3 &= rec_bits(lib, c_b, c_w, B.w23 >> 16);
            }
            bool ovf = hit && !inl;
            while (__any_sync(kFull, ovf)) {          // cold (a loop, so that it stays a branch): classes in overflow form
                if (ovf) {
#pragma unroll 1
                    for (int j = 0; j < na; j++) {
                        const uint32_t word = j == 0 ? (B.w01 & 0xFFFFu) : (j == 1 ? (B.w01 >> 16) : (j == 2 ? (B.w23 & 0xFFFFu) : (B.w23 >> 16)));
                        const uint32_t v = rec_lookup_overflow(lib.ov_w, lib.ov_b, c_b.x, c_b.y, word);
                        if (j == 0) B.a0 &= v; else if (j == 1) B.a1 &= v; else if (j == 2) B.a2 &= v; else B.a3 &= v;
                    }
                }
                ovf = false;
            }
        }
    } else if (!intersect_generic(lib, lw, lb, na, hit, c_b, c_w, lane)) {
        dead = true;
    }
    return true;
}

template <bool kStats>
__device__ __forceinline__ bool probe_mate(const LibDev &lib, const ReadsDev &R, uint64_t read, int lane, uint32_t cap,
                                           List *lists /* [2] */, MateProbe &M, uint32_t &n_probe, uint32_t &slots_read) {
    const uint8_t *rec = R.packed + read * R.stride;
    const int W = (int)R.words;
    const int L = read_length(R, read);
    const int k = lib.k;
    const int P = L - k + 1;
    M.L = L; M.P = P;
    const uint32_t kmask_lo = (uint32_t)lib.kmask, kmask_hi = (uint32_t)(lib.kmask >> 32), kbits = (uint32_t)lib.kbits;
    const int rshift = 64 - 2 * k;                          // revcomp: bits to drop after the 64-bit reversal
    const uint32_t nb = lib.n_buckets;
    uint32_t nh0 = 0, nh1 = 0;
    int seed_i0 = -1, seed_i1 = -1;
    int na0 = -1, na1 = -1, owner = -1;                      // pairs of B per orientation (-1: no hit yet); register owner
    bool dead0 = false, dead1 = false;                      // B already empty (lists in memory only)
    OwnerB B;
    B.w01 = B.w23 = 0xFFFFFFFFu; B.b0 = B.b1 = B.b2 = B.b3 = 0; B.a0 = B.a1 = B.a2 = B.a3 = kFull;
    // the packed read: lane t holds sequence word t (two 32-bit halves) and N-mask word t; rounds fetch them by shuffle
    uint32_t my_lo = 0, my_hi = 0, my_n = 0;
    if (lane < W && P > 0) {
        const uint2 v = *reinterpret_cast<const uint2 *>(rec + (size_t)lane * 8);
        my_lo = v.x; my_hi = v.y;
        my_n = *reinterpret_cast<const uint32_t *>(rec + (size_t)W * 8 + (size_t)lane * 4);
    }
    uint32_t w0 = __shfl_sync(kFull, my_lo, 0), w1 = __shfl_sync(kFull, my_hi, 0), n_lo = __shfl_sync(kFull, my_n, 0);
    const bool upper = lane >= 16;
    const int n_rounds = P > 0 ? (P + 31) >> 5 : 0;

#pragma unroll 1
    for (int r = 0; r < n_rounds; r++) {
        const int i = (r << 5) + lane;
        // ---- k-mer x at position i and its reverse complement y, as 32-bit halves ---------------------
        const uint32_t w2 = __shfl_sync(kFull, my_lo, r + 1), w3 = __shfl_sync(kFull, my_hi, r + 1), n_hi = __shfl_sync(kFull, my_n, r + 1);
        const uint32_t ea = upper ? w1 : w0, eb = upper ? w2 : w1, ec = upper ? w3 : w2;
        const uint32_t x_lo = __funnelshift_r(ea, eb, 2 * lane) & kmask_lo;      // funnel shifts take the amount modulo 32
        const uint32_t x_hi = __funnelshift_r(eb, ec, 2 * lane) & kmask_hi;
        const bool valid = i < P && (__funnelshift_r(n_lo, n_hi, lane) & kbits) == 0;
        w0 = w2; w1 = w3; n_lo = n_hi;
        uint32_t p_lo = __brev(~x_hi), p_hi = __brev(~x_lo);                    // 64-bit bit reversal of the complement
        p_lo = ((p_lo >> 1) & 0x55555555u) | ((p_lo << 1) & 0xAAAAAAAAu);        // bits of a base back in order
        p_hi = ((p_hi >> 1) & 0x55555555u) | ((p_hi << 1) & 0xAAAAAAAAu);
        const uint32_t y_lo = rshift >= 32 ? p_hi >> (rshift - 32) : __funnelshift_r(p_lo, p_hi, rshift);
        const uint32_t y_hi = rshift >= 32 ? 0u : p_hi >> rshift;
        const bool x_lt = x_hi < y_hi || (x_hi == y_hi && x_lo < y_lo), x_eq = x_hi == y_hi && x_lo == y_lo;
        const uint32_t c_lo = x_lt ? x_lo : y_lo, c_hi = x_lt ? x_hi : y_hi;
        // ---- table: first bucket always (lanes without a k-mer read bucket 0: one shared sector) -----------
        const uint32_t mix = kmer_mix(c_lo, c_hi);
        const uint32_t b1 = valid ? kmer_bucket1(mix, nb) : 0u;
        uint4 e_lo, e_hi;
        ldg256(lib.table + 2 * (size_t)b1, e_lo, e_hi);
        bool m0 = e_lo.x == c_lo && e_lo.y == c_hi, m1 = e_hi.x == c_lo && e_hi.y == c_hi;
        const bool need2 = valid && !(m0 || m1) && (e_lo.z & kDevSpill);
        if (kStats) { n_probe += valid ? 1u : 0u; slots_read += (valid ? 1u : 0u) + (need2 ? 1u : 0u); }
        // own-strand info belongs to orientation 0 when x is the canonical form (x <= y), to orientation 1 when y is
        const bool xs = x_lt || x_eq, ys = !x_lt;
        uint32_t ecls = m0 ? e_lo.z : e_hi.z;
        bool found = valid && (m0 || m1);
        uint32_t cl0 = (found && xs != ((ecls & kDevRc) != 0)) ? (ecls & kDevIdMask) : kInvalid;
        uint32_t cl1 = (found && ys != ((ecls & kDevRc) != 0)) ? (ecls & kDevIdMask) : kInvalid;
        // cold (a loop, so that it stays a branch): the key may sit in its second bucket, or the k-mer is present on both
        // strands of the library (dual record)
        bool slow = need2 || (found && (ecls & kDevDual));
        while (__any_sync(kFull, slow)) {
            if (slow) {
                if (need2) {
                    ldg256(lib.table + 2 * (size_t)kmer_bucket2(mix, c_lo, b1, nb), e_lo, e_hi);
                    m0 = e_lo.x == c_lo && e_lo.y == c_hi; m1 = e_hi.x == c_lo && e_hi.y == c_hi;
                    found = m0 || m1;
                    ecls = m0 ? e_lo.z : e_hi.z;
                    cl0 = (found && xs != ((ecls & kDevRc) != 0)) ? (ecls & kDevIdMask) : kInvalid;
                    cl1 = (found && ys != ((ecls & kDevRc) != 0)) ? (ecls & kDevIdMask) : kInvalid;
                }
                if (found && (ecls & kDevDual)) {
                    const uint4 d = __ldg(lib.dual + (ecls & kDevIdMask));
                    cl0 = xs ? d.x : d.z;
                    cl1 = ys ? d.x : d.z;
                }
            }
            slow = false;
        }
        // ---- hit counts, seeds, candidate sets --------------------------------------------------------------------
        // orientation 0 reads left to right: its seed is the FIRST hit; the reverse complement visits the positions
        // right to left: its first hit is the LAST one here
        const unsigned hb0 = __ballot_sync(kFull, cl0 != kInvalid), hb1 = __ballot_sync(kFull, cl1 != kInvalid);
        if (hb0) {
            nh0 += __popc(hb0);
            if (seed_i0 < 0) seed_i0 = (r << 5) + __ffs(hb0) - 1;
            if (!dead0 && !candidate_round(lib, 0, cl0, cap, lane, lists[0].w, lists[0].b, na0, owner, dead0, B)) return false;
        }
        if (hb1) {
            nh1 += __popc(hb1);
            seed_i1 = P - 1 - ((r << 5) + 31 - __clz(hb1));
            if (!dead1 && !candidate_round(lib, 1, cl1, cap, lane, lists[1].w, lists[1].b, na1, owner, dead1, B)) return false;
        }
    }
    // lists in memory are complete; owner: one REDUX per word of B for the whole read, B stays in registers (M.reg)
    lists[0].n = na0 > 0 ? na0 : 0; lists[1].n = na1 > 0 ? na1 : 0;
    M.owner = owner;
    if (owner >= 0) {
        const int na = owner ? na1 : na0;
        M.reg.w01 = B.w01; M.reg.w23 = B.w23;
        M.reg.b0 = B.b0 & __reduce_and_sync(kFull, B.a0);
        M.reg.b1 = na > 1 ? B.b1 & __reduce_and_sync(kFull, B.a1) : 0u;
        M.reg.b2 = na > 2 ? B.b2 & __reduce_and_sync(kFull, B.a2) : 0u;
        M.reg.b3 = na > 3 ? B.b3 & __reduce_and_sync(kFull, B.a3) : 0u;
    }
    __syncwarp();
    M.nh[0] = nh0; M.nh[1] = nh1; M.seed_i[0] = seed_i0; M.seed_i[1] = seed_i1;
    return true;
}

// the owner's candidate set -> its list in memory (callers that keep working on lists: wide_kernel)
__device__ __forceinline__ void owner_to_list(const MateProbe &M, List *lists, int lane) {
    if (M.owner < 0) return;
    List &Lo = lists[M.owner];
    if (lane < Lo.n) {
        Lo.w[lane] = lane == 0 ? (M.reg.w01 & 0xFFFFu) : (lane == 1 ? (M.reg.w01 >> 16) : (lane == 2 ? (M.reg.w23 & 0xFFFFu) : (M.reg.w23 >> 16)));
        Lo.b[lane] = lane == 0 ? M.reg.b0 : (lane == 1 ? M.reg.b1 : (lane == 2 ? M.reg.b2 : M.reg.b3));
    }
    __syncwarp();
}

// SW work items of one partial orientation: candidates in ascending reference order.  Lane = CANDIDATE (the t-th set
// bit over the words of B), not word: allele-family sets have 1-4 words and a dozen members, so a lane-per-word loop
// would run one or two lanes through all of them (measured: 1.5 threads per instruction).
__device__ __forceinline__ void emit_items(const LibDev &lib, const List &B, uint32_t seed_cls, uint32_t seed_off, int seed_i,
                                           uint32_t ro_idx, uint32_t len, uint32_t cnt, SwItem *items, uint32_t off, int lane) {
    const Rec seed = load_rec(lib, seed_cls);
    uint32_t run = 0;
    for (int base = 0; base < B.n; base += 32) {
        const int j = base + lane;
        const uint32_t bits = j < B.n ? B.b[j] : 0u, word = j < B.n ? B.w[j] : 0u;
        uint32_t tot;
        const uint32_t ex = warp_excl_scan(__popc(bits), lane, tot);        // candidates before word j (within this chunk of words)
        const int nw = min(32, B.n - base);
        for (uint32_t c0 = 0; c0 < tot; c0 += 32) {
            const uint32_t c = c0 + lane;                                    // candidate index within the chunk
            int owner = 0;
            for (int jj = 1; jj < nw; jj++) if (__shfl_sync(kFull, ex, jj) <= c) owner = jj;     // last word that starts at or before c
            const uint32_t obits = __shfl_sync(kFull, bits, owner), oword = __shfl_sync(kFull, word, owner);
            const uint32_t oex = __shfl_sync(kFull, ex, owner);
            if (c < tot) {
                uint32_t rest = obits;
                for (uint32_t t = c - oex; t > 0; t--) rest &= rest - 1;     // drop the candidates below mine
                const uint32_t r = oword * 32 + (uint32_t)(__ffs(rest) - 1);
                const uint32_t pos = __ldg(lib.positions + seed_off + rec_rank(lib, seed, r));
                SwItem it;
                it.ro = ro_idx | (len << kRoIdxBits); it.ref = r;
                it.gwin = __ldg(lib.ref_gstart + r) + pos - (uint32_t)seed_i - (uint32_t)kBand;
                it.v = 0;
                items[off + run + c] = it;
            }
        }
        run += tot;
    }
    if (lane == 0 && (cnt & 1)) {
        SwItem it; it.ro = ro_idx | (len << kRoIdxBits); it.ref = kInvalid; it.gwin = 0; it.v = 0;
        items[off + cnt] = it;
    }
}

__device__ __forceinline__ void carve_scratch(uint32_t *s, uint32_t cap, List *L4, List &T, List &Bst) {
#pragma unroll
    for (int q = 0; q < 4; q++) { L4[q].w = s + (size_t)q * 2 * cap; L4[q].b = L4[q].w + cap; L4[q].n = 0; }
    T.w = s + (size_t)8 * cap; T.b = T.w + 2 * (size_t)cap; T.n = 0;
    Bst.w = s + (size_t)12 * cap; Bst.b = Bst.w + 2 * (size_t)cap; Bst.n = 0;
}

// ---------------------------------------------------------------------------------------------
// X3a/X3b kernel: one warp per read (pair).  Probes the table and intersects the classes; leaves one 32-byte summary
// per mate and orientation (OriSum).  Scoring / filtering / feature calling is NOT done here: that logic is scalar per
// read, so it runs one THREAD per read in call_fast_kernel (a warp per read would idle 31 lanes on it), and only the
// reads that need Smith-Waterman or carry wide candidate sets take the warp-per-read call_slow_kernel.
// Wide reads (narrowest class wider than the shared-memory lists) go to wide_kernel.
// Single-end batches run probe_thread_kernel first; this warp form then takes only the reads it listed
// (probe_list_kernel).  Paired-end batches and NB200_PROBE_WARP=1 run probe_kernel on every read.
// ---------------------------------------------------------------------------------------------
template <int NM, bool kStats>       // mates per read; kStats: count lookups / sectors (nb200_set_stats)
__device__ __forceinline__ void probe_read(const LibDev &lib, const ReadsDev &r1, const ReadsDev &r2, uint64_t read0, uint32_t gw,
                                           OriSum *__restrict__ sums, uint32_t *__restrict__ roB, uint32_t *__restrict__ wide_list,
                                           Counters *__restrict__ ctr, List *L4, int lane, uint32_t &n_probe, uint32_t &slots_read) {
    const uint64_t read = read0 + gw;
    constexpr int n_ro = NM * 2;
    bool wide = false;
#pragma unroll
    for (int m = 0; m < NM; m++) {
        if (wide) break;
        MateProbe M;
        if (!probe_mate<kStats>(lib, m ? r2 : r1, read, lane, lib.narrow_cap, &L4[m * 2], M, n_probe, slots_read)) { wide = true; break; }
#pragma unroll
        for (int o = 0; o < 2; o++) {
            const int q = m * 2 + o;
            const int na = L4[q].n;
            const bool in_mem = na > 4, reg = M.owner == o;
            const bool full = M.nh[o] && (int)M.nh[o] == M.P;
            // words 0-1: nh | seed_i << 16,  na | flags << 8 | len << 16;  words 2-7: w01, w23, b0..b3
            uint32_t w01 = 0xFFFFFFFFu, w23 = 0xFFFFFFFFu, b0 = 0, b1 = 0, b2 = 0, b3 = 0;
            if (reg) { w01 = M.reg.w01; w23 = M.reg.w23; b0 = M.reg.b0; b1 = M.reg.b1; b2 = M.reg.b2; b3 = M.reg.b3; }
            else if (na > 0 && !in_mem) {                       // second orientation of a read that hits on both strands: from its list
                const uint32_t *lw = L4[q].w, *lb = L4[q].b;
                const uint32_t x0 = lw[0], x1 = na > 1 ? lw[1] : 0xFFFFu, x2 = na > 2 ? lw[2] : 0xFFFFu, x3 = na > 3 ? lw[3] : 0xFFFFu;
                w01 = x0 | (x1 << 16); w23 = x2 | (x3 << 16);
                b0 = lb[0]; b1 = na > 1 ? lb[1] : 0u; b2 = na > 2 ? lb[2] : 0u; b3 = na > 3 ? lb[3] : 0u;
            } else if (in_mem) {                                // wide candidate set: park it in the list area, read-indexed
                uint32_t *dst = roB + ((size_t)gw * n_ro + q) * 2 * kCap;
                for (int j = lane; j < na; j += 32) { dst[j] = L4[q].w[j]; dst[kCap + j] = L4[q].b[j]; }
            }
            if (lane == 0) {
                uint4 *dst = reinterpret_cast<uint4 *>(sums + (size_t)gw * n_ro + q);
                const uint32_t flags = (full ? kSumFull : 0u) | (in_mem ? kSumInMem : 0u);
                dst[0] = make_uint4((M.nh[o] & 0xFFFFu) | ((uint32_t)(M.seed_i[o] & 0xFFFF) << 16),
                                    (uint32_t)na | (flags << 8) | ((uint32_t)M.L << 16), w01, w23);
                dst[1] = make_uint4(b0, b1, b2, b3);
            }
        }
    }
    if (wide && lane == 0) {
        wide_list[atomicAdd(&ctr->n_wide, 1ull)] = gw;
        reinterpret_cast<uint4 *>(sums + (size_t)gw * n_ro)[0] = make_uint4(0u, (uint32_t)kSumWide << 8, 0xFFFFFFFFu, 0xFFFFFFFFu);
    }
}

template <bool kStats>
__device__ __forceinline__ void add_probe_stats(Counters *ctr, int lane, uint32_t n_probe, uint32_t slots_read) {
    if (!kStats) return;
    n_probe = warp_sum(n_probe);
    slots_read = warp_sum(slots_read);
    if (lane == 0 && n_probe) {
        atomicAdd(&ctr->probes[blockIdx.x & (kCtrSpread - 1)], (unsigned long long)n_probe);
        atomicAdd(&ctr->probe_slots[blockIdx.x & (kCtrSpread - 1)], (unsigned long long)slots_read);
    }
}

__device__ __forceinline__ void carve_probe_lists(uint32_t *smem, int wib, List *L4) {
#pragma unroll
    for (int q = 0; q < 4; q++) { L4[q].w = smem + ((size_t)wib * 4 + q) * 2 * kCap; L4[q].b = L4[q].w + kCap; L4[q].n = 0; }
}

template <int NM, bool kStats>
__global__ void __launch_bounds__(kProbeWarps * 32, (NM == 2 ? 24 : 36) / kProbeWarps)
probe_kernel(LibDev lib, ReadsDev r1, ReadsDev r2, uint64_t read0, uint64_t n_reads, OriSum *__restrict__ sums,
             uint32_t *__restrict__ roB, uint32_t *__restrict__ wide_list, Counters *__restrict__ ctr) {
    __shared__ uint32_t smem[kProbeWarps * 4 * 2 * kCap];          // per warp: four lists (generic path only)
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const uint32_t gw = blockIdx.x * kProbeWarps + wib;            // a batch is at most 2^21 reads
    if (gw >= n_reads) return;
    List L4[4];
    carve_probe_lists(smem, wib, L4);
    uint32_t n_probe = 0, slots_read = 0;
    probe_read<NM, kStats>(lib, r1, r2, read0, gw, sums, roB, wide_list, ctr, L4, lane, n_probe, slots_read);
    add_probe_stats<kStats>(ctr, lane, n_probe, slots_read);
}

// The reads probe_thread_kernel listed (ctr->n_probe_warp of them): the warp form above, one warp per read over a
// grid-stride loop, with its anchor rule, wide-path decision and wide_list unchanged.  Single-end only.
constexpr int kProbeListBlocks = 24 / kProbeWarps;   // per SM: 85 registers for the grid-stride loop, no spills
template <bool kStats>
__global__ void __launch_bounds__(kProbeWarps * 32, kProbeListBlocks)
probe_list_kernel(LibDev lib, ReadsDev r1, uint64_t read0, const uint32_t *__restrict__ warp_list, OriSum *__restrict__ sums,
                  uint32_t *__restrict__ roB, uint32_t *__restrict__ wide_list, Counters *__restrict__ ctr) {
    __shared__ uint32_t smem[kProbeWarps * 4 * 2 * kCap];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const uint32_t n = (uint32_t)ctr->n_probe_warp;
    List L4[4];
    carve_probe_lists(smem, wib, L4);
    uint32_t n_probe = 0, slots_read = 0;
    for (uint32_t t = blockIdx.x * kProbeWarps + wib; t < n; t += gridDim.x * kProbeWarps) {
        __syncwarp();                                              // the previous read's lists are no longer read
        probe_read<1, kStats>(lib, r1, r1, read0, warp_list[t], sums, roB, wide_list, ctr, L4, lane, n_probe, slots_read);
    }
    add_probe_stats<kStats>(ctr, lane, n_probe, slots_read);
}

// ---------------------------------------------------------------------------------------------
// X3a + X3b, one THREAD per single-end read: the thread walks its read's k-mer positions in order.
//
// The k-mer and its reverse complement roll along the read one base at a time (64-bit words, 2 bits per base); a
// k-mer is valid when the last N base lies before it.  The lookup is that of probe_mate and host_lookup (canonical
// form, kmer_mix, one 256-bit load of the first bucket; second bucket and dual records on a cold branch).  Positions
// go in groups of kProbeGroup: the group's bucket loads, then its class-record loads, are issued before the first is
// used.  On a B200 a larger group bought nothing: its registers cost occupancy, and the kernel's speed follows the
// number of resident warps (cfg2 probe time, 10 M reads: 8.0 / 8.4 / 9.7 / 12.8 / 22.5 ms for groups of 1 / 2 / 3 / 4 / 8,
// before the candidate sets moved to shared memory).  So the group is 1 and the register budget is what is tuned.
//
// Candidate set per orientation (hit count, previous class and seed in registers, B in shared memory): B is anchored
// on the orientation's FIRST hit class and every later hit class is ANDed in.  A hit whose class id equals the previous hit's in that orientation skips the record load and the
// AND (AND is idempotent; runs of one class are the normal case for allele families).  B only shrinks, so its members
// do not depend on the anchor: OriSum differs from probe_kernel's only in which (empty) words B keeps.
//
// A read whose anchor is an overflow-form record or has more than min(4, narrow_cap) words is appended to warp_list
// (one atomic per warp) and nothing else is written for it: probe_list_kernel probes it as probe_kernel would, and
// counts its lookups, so the kStats counters equal probe_kernel's.
// ---------------------------------------------------------------------------------------------
constexpr int kProbeThreads = 128;
constexpr int kProbeGroup = 1;
constexpr int kProbeThreadBlocks = 10;   // blocks per SM: 47 registers, no spills (12 blocks: 40 registers, spills, slower)

struct ThreadB {                 // one orientation, in registers: hits, previous hit class, seed
    uint32_t nh, prev;
    int seed;                    // orientation 0: first hit position; orientation 1: last
};
// The rest of an orientation's state lives in shared memory, one column per thread (conflict-free), because it is only
// touched when the class changes: registers decide the kernel's occupancy, and occupancy its speed.
enum { SB_NA = 0, SB_W01, SB_W23, SB_B0, SB_B1, SB_B2, SB_B3, SB_N };
#define NB200_SB(f) sb[(f) * kProbeThreads]

// one hit of class `cl` at position i in orientation o; (c_b, c_w) is its record when `cl` differs from the previous hit
// class (loaded by the caller).  Returns false when the read must take the warp form.
__device__ __forceinline__ bool thread_hit(const LibDev &lib, ThreadB &T, uint32_t *sb, uint32_t cl, int i, int o, uint32_t cap,
                                           const uint4 c_b, const uint4 c_w) {
    T.nh++;
    if (o == 0) T.seed = T.seed < 0 ? i : T.seed; else T.seed = i;
    if (cl == T.prev) return true;
    const bool inl = (int32_t)c_w.z >= 0;
    if (T.prev == kInvalid) {                                      // anchor
        T.prev = cl;
        const uint32_t na = c_w.z & 0xFFu;
        NB200_SB(SB_NA) = na;
        if (!inl || na > cap) return false;
        NB200_SB(SB_W01) = c_w.x; NB200_SB(SB_W23) = c_w.y;
        NB200_SB(SB_B0) = c_b.x; NB200_SB(SB_B1) = c_b.y; NB200_SB(SB_B2) = c_b.z; NB200_SB(SB_B3) = c_b.w;
        return true;
    }
    T.prev = cl;
    const uint32_t w01 = NB200_SB(SB_W01), w23 = NB200_SB(SB_W23);
    uint4 m = c_b;                                                 // same reference words: word by word
    if (!(inl && c_w.x == w01 && c_w.y == w23)) {                  // unused words of B (0xFFFF) are zeroed at the end
        m.x = rec_bits(lib, c_b, c_w, w01 & 0xFFFFu);
        m.y = rec_bits(lib, c_b, c_w, w01 >> 16);
        m.z = rec_bits(lib, c_b, c_w, w23 & 0xFFFFu);
        m.w = rec_bits(lib, c_b, c_w, w23 >> 16);
    }
    NB200_SB(SB_B0) &= m.x; NB200_SB(SB_B1) &= m.y; NB200_SB(SB_B2) &= m.z; NB200_SB(SB_B3) &= m.w;
    return true;
}

template <bool kStats>
__global__ void __launch_bounds__(kProbeThreads, kProbeThreadBlocks)
probe_thread_kernel(LibDev lib, ReadsDev R, uint64_t read0, uint64_t n_reads, OriSum *__restrict__ sums,
                    uint32_t *__restrict__ warp_list, Counters *__restrict__ ctr) {
    const uint32_t gr = blockIdx.x * kProbeThreads + threadIdx.x;   // a batch is at most 2^21 reads
    const bool active = gr < n_reads;
    const uint64_t read = read0 + (active ? gr : 0u);
    const uint8_t *rec = R.packed + read * R.stride;
    const uint64_t *seq = reinterpret_cast<const uint64_t *>(rec);
    const int W = (int)R.words, k = lib.k;
    const int P = (active ? read_length(R, read) : 0) - k + 1;
    const uint64_t kmask = lib.kmask;
    const int top = 2 * k - 2;                                     // bit of the newest base in the forward k-mer
    const uint32_t nb = lib.n_buckets, cap = min(4u, lib.narrow_cap);
    __shared__ uint32_t s_b[2 * SB_N * kProbeThreads];
    uint32_t *const sb0 = s_b + threadIdx.x, *const sb1 = sb0 + SB_N * kProbeThreads;
    ThreadB T[2];
#pragma unroll
    for (int o = 0; o < 2; o++) {
        uint32_t *sb = o ? sb1 : sb0;
        T[o].nh = 0; T[o].prev = kInvalid; T[o].seed = -1;
        NB200_SB(SB_NA) = 0; NB200_SB(SB_W01) = NB200_SB(SB_W23) = 0xFFFFFFFFu;
        NB200_SB(SB_B0) = NB200_SB(SB_B1) = NB200_SB(SB_B2) = NB200_SB(SB_B3) = 0;
    }
    uint32_t n_probe = 0, slots_read = 0;
    bool fallback = false;
    // base stream: `cur` holds the packed word of base p onwards, `ncur` its N bits
    uint64_t cur = 0, x = 0, y = 0;
    uint32_t ncur = 0;
    int p = 0, last_n = -1;
    auto push_base = [&]() {
        if ((p & 31) == 0) {
            const int w = p >> 5;
            cur = w < W ? seq[w] : 0ull;
            ncur = w < W ? reinterpret_cast<const uint32_t *>(seq + W)[w] : 0u;   // N masks follow the sequence words
        }
        const uint32_t b = (uint32_t)cur & 3u;
        last_n = (ncur & 1u) ? p : last_n;
        cur >>= 2; ncur >>= 1;
        x = (x >> 2) | ((uint64_t)b << top);
        y = ((y << 2) | (b ^ 3u)) & kmask;
        p++;
    };
    if (P > 0)
        for (int t = 0; t < k - 1; t++) push_base();
#pragma unroll 1
    for (int i0 = 0; i0 < P; i0 += kProbeGroup) {
        uint32_t c_lo[kProbeGroup], c_hi[kProbeGroup];
        bool valid[kProbeGroup], xs[kProbeGroup], ys[kProbeGroup];
        uint4 e_lo[kProbeGroup], e_hi[kProbeGroup];
#pragma unroll
        for (int g = 0; g < kProbeGroup; g++) {
            push_base();
            const int i = i0 + g;
            valid[g] = i < P && last_n < i;
            const bool x_lt = x < y;
            xs[g] = x <= y; ys[g] = !x_lt;
            const uint64_t c = x_lt ? x : y;
            c_lo[g] = (uint32_t)c; c_hi[g] = (uint32_t)(c >> 32);
            e_lo[g] = make_uint4(kInvalid, kInvalid, 0u, 0u); e_hi[g] = e_lo[g];
            if (valid[g]) ldg256(lib.table + 2 * (size_t)kmer_bucket1(kmer_mix(c_lo[g], c_hi[g]), nb), e_lo[g], e_hi[g]);
        }
        uint32_t cl0[kProbeGroup], cl1[kProbeGroup];
#pragma unroll
        for (int g = 0; g < kProbeGroup; g++) {
            const uint32_t clo = c_lo[g], chi = c_hi[g];
            bool m0 = e_lo[g].x == clo && e_lo[g].y == chi, m1 = e_hi[g].x == clo && e_hi[g].y == chi;
            uint32_t ecls = m0 ? e_lo[g].z : e_hi[g].z;
            bool found = valid[g] && (m0 || m1);
            const bool need2 = valid[g] && !(m0 || m1) && (e_lo[g].z & kDevSpill);
            if (kStats) { n_probe += valid[g] ? 1u : 0u; slots_read += (valid[g] ? 1u : 0u) + (need2 ? 1u : 0u); }
            if (need2 || (found && (ecls & kDevDual))) {           // cold: the key's second bucket, or a dual record
                if (need2) {
                    const uint32_t mix = kmer_mix(clo, chi);
                    uint4 f_lo, f_hi;
                    ldg256(lib.table + 2 * (size_t)kmer_bucket2(mix, clo, kmer_bucket1(mix, nb), nb), f_lo, f_hi);
                    m0 = f_lo.x == clo && f_lo.y == chi; m1 = f_hi.x == clo && f_hi.y == chi;
                    found = m0 || m1;
                    ecls = m0 ? f_lo.z : f_hi.z;
                }
                cl0[g] = (found && xs[g] != ((ecls & kDevRc) != 0)) ? (ecls & kDevIdMask) : kInvalid;
                cl1[g] = (found && ys[g] != ((ecls & kDevRc) != 0)) ? (ecls & kDevIdMask) : kInvalid;
                if (found && (ecls & kDevDual)) {
                    const uint4 d = __ldg(lib.dual + (ecls & kDevIdMask));
                    cl0[g] = xs[g] ? d.x : d.z;
                    cl1[g] = ys[g] ? d.x : d.z;
                }
            } else {
                cl0[g] = (found && xs[g] != ((ecls & kDevRc) != 0)) ? (ecls & kDevIdMask) : kInvalid;
                cl1[g] = (found && ys[g] != ((ecls & kDevRc) != 0)) ? (ecls & kDevIdMask) : kInvalid;
            }
        }
        // the class records the group needs (a class that differs from the previous hit class of its orientation), all
        // loads issued before the first is used: one per position, orientation 0 first.  Both orientations hit with
        // different classes only through dual records; orientation 1's record is then loaded on its own.
        uint4 r_b[kProbeGroup], r_w[kProbeGroup];
        uint32_t r_cl[kProbeGroup];
        {
            uint32_t p0 = T[0].prev, p1 = T[1].prev;
#pragma unroll
            for (int g = 0; g < kProbeGroup; g++) {
                const bool n0 = cl0[g] != kInvalid && cl0[g] != p0, n1 = cl1[g] != kInvalid && cl1[g] != p1;
                r_cl[g] = n0 ? cl0[g] : (n1 ? cl1[g] : kInvalid);
                if (cl0[g] != kInvalid) p0 = cl0[g];
                if (cl1[g] != kInvalid) p1 = cl1[g];
                r_b[g] = make_uint4(0u, 0u, 0u, 0u); r_w[g] = r_b[g];
                if (r_cl[g] != kInvalid) ldg256_cached(lib.class_rec + 2 * (size_t)r_cl[g], r_b[g], r_w[g]);
            }
        }
#pragma unroll
        for (int g = 0; g < kProbeGroup; g++) {
            if (cl0[g] != kInvalid && !thread_hit(lib, T[0], sb0, cl0[g], i0 + g, 0, cap, r_b[g], r_w[g])) fallback = true;
            if (cl1[g] != kInvalid) {
                uint4 c_b = r_b[g], c_w = r_w[g];
                if (cl1[g] != T[1].prev && cl1[g] != r_cl[g]) ldg256_cached(lib.class_rec + 2 * (size_t)cl1[g], c_b, c_w);
                if (!thread_hit(lib, T[1], sb1, cl1[g], i0 + g, 1, cap, c_b, c_w)) fallback = true;
            }
        }
        if (fallback) break;
    }
    // the reads left to the warp form: one atomic per warp
    const unsigned fb = __ballot_sync(kFull, active && fallback);
    if (fb) {
        const int lane = threadIdx.x & 31, leader = __ffs(fb) - 1;
        uint32_t base = 0;
        if (lane == leader) base = (uint32_t)atomicAdd(&ctr->n_probe_warp, (unsigned long long)__popc(fb));
        base = __shfl_sync(kFull, base, leader);
        if (active && fallback) warp_list[base + __popc(fb & ((1u << lane) - 1))] = gr;
    }
    if (fallback) n_probe = slots_read = 0;                        // probe_list_kernel counts the read
    add_probe_stats<kStats>(ctr, threadIdx.x & 31, n_probe, slots_read);
    if (!active || fallback) return;
    uint4 *dst = reinterpret_cast<uint4 *>(sums + (size_t)gr * 2);
#pragma unroll
    for (int o = 0; o < 2; o++) {
        const ThreadB &B = T[o];
        const uint32_t *sb = o ? sb1 : sb0;
        const uint32_t na = B.prev == kInvalid ? 0u : NB200_SB(SB_NA);
        const int seed = B.nh == 0 ? -1 : (o == 0 ? B.seed : P - 1 - B.seed);
        const uint32_t flags = (B.nh && (int)B.nh == P) ? kSumFull : 0u;
        dst[2 * o] = make_uint4((B.nh & 0xFFFFu) | ((uint32_t)(seed & 0xFFFF) << 16), na | (flags << 8) | ((uint32_t)(P + k - 1) << 16),
                                NB200_SB(SB_W01), NB200_SB(SB_W23));
        dst[2 * o + 1] = make_uint4(NB200_SB(SB_B0), na > 1 ? NB200_SB(SB_B1) : 0u, na > 2 ? NB200_SB(SB_B2) : 0u,
                                    na > 3 ? NB200_SB(SB_B3) : 0u);
    }
}
#undef NB200_SB

// ---------------------------------------------------------------------------------------------
// X4, one THREAD per read: every read whose orientations all resolved without alignment (no hit / empty class / every
// position hit) and whose candidate sets have at most 4 sparse words is scored, filtered and feature-called right here
// (DESIGN.md §2.5-2.6, same decisions as call_read).  The others are listed for call_slow_kernel.
// ---------------------------------------------------------------------------------------------
struct SmallList { uint32_t w[8], b[8]; int n; };

__device__ __forceinline__ void small_from_sum(const uint4 lo, const uint4 hi, SmallList &A) {
    A.n = (int)(lo.y & 0xFFu);
    A.w[0] = lo.z & 0xFFFFu; A.w[1] = lo.z >> 16; A.w[2] = lo.w & 0xFFFFu; A.w[3] = lo.w >> 16;
    A.b[0] = hi.x; A.b[1] = hi.y; A.b[2] = hi.z; A.b[3] = hi.w;
}
__device__ __forceinline__ uint32_t small_count(const SmallList &A) {
    uint32_t c = 0;
    for (int j = 0; j < A.n; j++) c += __popc(A.b[j]);
    return c;
}

// ---------------------------------------------------------------------------------------------
// X4 for one read by ONE thread (DESIGN.md §2.5-2.6, same decisions as the warp-cooperative call_read): status and
// score per orientation from (hits, candidates, best V), strand configurations, mate union / intersection on the
// inline candidate sets (lo / hi in the layout of OriSum: at most 4 sparse words), reference -> feature.  Writes the
// ten words of the nb200_read_result into rec and the feature ids (padded with -1 to max_hits) into fout; returns
// the number of features called.
// ---------------------------------------------------------------------------------------------
template <int NM>
__device__ __forceinline__ int thread_call(const LibDev &lib, const CallParams &cp, const uint4 (&lo)[NM * 2], const uint4 (&hi)[NM * 2],
                                           const uint32_t (&nh)[4], const uint32_t (&nc)[4], const int (&len)[4], const int (&vbest)[4],
                                           uint32_t n_sw, int32_t *fout, uint32_t *rec) {
    constexpr int n_ro = NM * 2;
    constexpr bool paired = NM == 2;
    const int mh = cp.max_hits;
    int n_feat = 0;
    // ---- per orientation: status / score ---------------------------------------------------------------------------
    int st[4] = {ST_NONE, ST_NONE, ST_NONE, ST_NONE}, sc[4] = {0, 0, 0, 0}, ed[4] = {0, 0, 0, 0};
#pragma unroll
    for (int o = 0; o < n_ro; o++) {
        if (nh[o] == 0) { st[o] = ST_NO_MATCH; continue; }
        if (vbest[o] < 0) { st[o] = ST_EMPTY; continue; }
        sc[o] = (vbest[o] + kVW - 1) / kVW;                          // V = 64 score - edits (exact containment: V = 64 L)
        ed[o] = sc[o] * kVW - vbest[o];
        if (sc[o] < cp.score_threshold) st[o] = ST_SCORE;
        else if (sc[o] < (int)cp.min_score[len[o]]) st[o] = ST_PERCENT;
        else if (cp.discard_multiple_matches && nc[o] > 1) st[o] = ST_MULTI;
        else st[o] = ST_PASS;
    }
    const bool any_pass = st[0] == ST_PASS || st[1] == ST_PASS || st[2] == ST_PASS || st[3] == ST_PASS;
    int chosen = -1, chosen_max = 0;
    int first_fail = (!any_pass && paired && cp.require_valid_pair) ? RS_NOT_VALID_PAIR : RS_NO_PASS;
    uint32_t chosen_score = 0;
    int reason, n_feat_local = 0;
    if constexpr (!paired) {
        // single-end: configuration F = orientation 0, R = orientation 1 (in this order; the higher score wins, ties -> F);
        // everything below indexes registers statically
        const bool en0 = any_pass && cp.strand_filter != NB200_THREEPRIME, en1 = any_pass && cp.strand_filter != NB200_FIVEPRIME;
        if (en0 && st[0] == ST_PASS) { chosen = 0; chosen_score = (uint32_t)sc[0]; }
        if (en1 && st[1] == ST_PASS && (chosen < 0 || (uint32_t)sc[1] > chosen_score)) { chosen = 1; chosen_score = (uint32_t)sc[1]; }
        chosen_max = (int)chosen_score;
        reason = first_fail;
        if (chosen >= 0) {
            const uint4 l = chosen ? lo[1] : lo[0], h = chosen ? hi[1] : hi[0];
            const int n = (int)(l.y & 0xFFu);
            const uint32_t w0 = l.z & 0xFFFFu, w1 = l.z >> 16, w2 = l.w & 0xFFFFu, w3 = l.w >> 16;
            const uint32_t b0 = h.x, b1 = n > 1 ? h.y : 0u, b2 = n > 2 ? h.z : 0u, b3 = n > 3 ? h.w : 0u;
            if (chosen_max < cp.score_filter) reason = RS_SCORE_FILTER;
            else {
                // features of the members in ascending order; with an identity map the feature IS the reference
                const bool ident = lib.identity != 0;
                int nf = 0;
                uint32_t prev = kInvalid;
                auto count_word = [&](uint32_t w, uint32_t bits) {
                    if (ident) { nf += __popc(bits); return; }
                    while (bits) {
                        const int bpos = __ffs(bits) - 1; bits &= bits - 1;
                        const uint32_t f = __ldg(lib.ref_feature + w * 32 + bpos);
                        if (f != prev) { nf++; prev = f; }
                    }
                };
                count_word(w0, b0); count_word(w1, b1); count_word(w2, b2); count_word(w3, b3);
                if (cp.discard_multi_hits > 0 && nf > cp.discard_multi_hits) reason = RS_MULTI_HITS;
                else if (nf > mh) reason = RS_MAX_HITS;
                else {
                    reason = RS_CALLED; n_feat_local = nf;
                    int at = 0;
                    prev = kInvalid;
                    auto emit_word = [&](uint32_t w, uint32_t bits) {
                        while (bits) {
                            const int bpos = __ffs(bits) - 1; bits &= bits - 1;
                            const uint32_t r = w * 32 + bpos;
                            const uint32_t f = ident ? r : __ldg(lib.ref_feature + r);
                            if (f != prev) { fout[at++] = (int32_t)f; prev = f; }
                        }
                    };
                    emit_word(w0, b0); emit_word(w1, b1); emit_word(w2, b2); emit_word(w3, b3);
                }
            }
        }
    } else {
    int order[4], n_cfg = 0;
    switch (any_pass ? cp.strand_filter : -1) {
    case -1: break;
    case NB200_FIVEPRIME: order[n_cfg++] = 0; break;
    case NB200_THREEPRIME: order[n_cfg++] = 1; break;
    case NB200_STRAND_NONE: order[n_cfg++] = 0; order[n_cfg++] = 1; order[n_cfg++] = 2; order[n_cfg++] = 3; break;
    default: order[n_cfg++] = 0; order[n_cfg++] = 1; break;
    }
    SmallList best;
    best.n = 0;
    for (int ci = 0; ci < n_cfg; ci++) {
        const int c = order[ci];
        const int ia = (c == 0 || c == 2) ? 0 : 1;            // F,FF: r1 fwd ; R,RR: r1 rc
        const int ib = (c == 0 || c == 3) ? 3 : 2;            // F,RR: r2 rc  ; R,FF: r2 fwd
        const int sa = sc[ia], sbv = sc[ib];
        const bool pa = st[ia] == ST_PASS, pb = st[ib] == ST_PASS;
        int fail = -1, maxmate = 0;
        uint32_t sum = 0;
        SmallList cur;
        cur.n = 0;
        if (cp.require_valid_pair && !(pa && pb)) fail = RS_NOT_VALID_PAIR;
        else if (!pa && !pb) fail = RS_NO_PASS;
        else if (pa && pb) {
            sum = (uint32_t)(sa + sbv); maxmate = max(sa, sbv);
            SmallList A, Bl;
            small_from_sum(lo[ia], hi[ia], A); small_from_sum(lo[ib], hi[ib], Bl);
            if (cp.intersect_level == 0) {                   // union (sorted merge)
                int i = 0, j = 0, n = 0;
                while (i < A.n || j < Bl.n) {
                    if (j >= Bl.n || (i < A.n && A.w[i] < Bl.w[j])) { cur.w[n] = A.w[i]; cur.b[n] = A.b[i]; i++; }
                    else if (i >= A.n || Bl.w[j] < A.w[i]) { cur.w[n] = Bl.w[j]; cur.b[n] = Bl.b[j]; j++; }
                    else { cur.w[n] = A.w[i]; cur.b[n] = A.b[i] | Bl.b[j]; i++; j++; }
                    n++;
                }
                cur.n = n;
            } else {
                uint32_t any = 0;
                for (int i = 0; i < A.n; i++) {
                    uint32_t v = 0;
                    for (int j = 0; j < Bl.n; j++) if (Bl.w[j] == A.w[i]) v = Bl.b[j];
                    cur.w[i] = A.w[i]; cur.b[i] = A.b[i] & v;
                    any |= cur.b[i];
                }
                cur.n = A.n;
                if (!any) {
                    if (cp.intersect_level >= 2) fail = RS_FORCE_INTERSECT;
                    else if (sbv > sa) cur = Bl; else cur = A;
                }
            }
        } else {
            if (cp.intersect_level >= 2) fail = RS_FORCE_INTERSECT;
            else { sum = (uint32_t)(pa ? sa : sbv); maxmate = (int)sum; small_from_sum(pa ? lo[ia] : lo[ib], pa ? hi[ia] : hi[ib], cur); }
        }
        if (fail >= 0) { if (ci == 0) first_fail = fail; continue; }
        if (chosen < 0 || sum > chosen_score) { chosen = c; chosen_score = sum; chosen_max = maxmate; best = cur; }
    }
    reason = first_fail;
    if (chosen >= 0) {
        if (chosen_max < cp.score_filter) reason = RS_SCORE_FILTER;
        else if (lib.identity) {
            const int nf = (int)small_count(best);
            if (cp.discard_multi_hits > 0 && nf > cp.discard_multi_hits) reason = RS_MULTI_HITS;
            else if (nf > mh) reason = RS_MAX_HITS;
            else {
                reason = RS_CALLED; n_feat_local = nf;
                int at = 0;
                for (int j = 0; j < best.n; j++) {
                    uint32_t bits = best.b[j];
                    while (bits) { const int bpos = __ffs(bits) - 1; bits &= bits - 1; fout[at++] = (int32_t)(best.w[j] * 32 + bpos); }
                }
            }
        } else {
            // references are ordered by feature: features of ascending members are non-decreasing
            int nf = 0;
            uint32_t prev = kInvalid;
            for (int j = 0; j < best.n; j++) {
                uint32_t bits = best.b[j];
                while (bits) {
                    const int bpos = __ffs(bits) - 1; bits &= bits - 1;
                    const uint32_t f = __ldg(lib.ref_feature + best.w[j] * 32 + bpos);
                    if (f != prev) { nf++; prev = f; }
                }
            }
            if (cp.discard_multi_hits > 0 && nf > cp.discard_multi_hits) reason = RS_MULTI_HITS;
            else if (nf > mh) reason = RS_MAX_HITS;
            else {
                reason = RS_CALLED; n_feat_local = nf;
                int at = 0;
                prev = kInvalid;
                for (int j = 0; j < best.n; j++) {
                    uint32_t bits = best.b[j];
                    while (bits) {
                        const int bpos = __ffs(bits) - 1; bits &= bits - 1;
                        const uint32_t f = __ldg(lib.ref_feature + best.w[j] * 32 + bpos);
                        if (f != prev) { fout[at++] = (int32_t)f; prev = f; }
                    }
                }
            }
        }
    }
    }   // paired
    n_feat = n_feat_local;
    for (int t = n_feat; t < mh; t++) fout[t] = -1;
    // the record, as 16-byte stores (layout of nb200_read_result)
    static_assert(sizeof(nb200_read_result) == 40 && offsetof(nb200_read_result, n_hits) == 8 && offsetof(nb200_read_result, n_cand) == 16 &&
                  offsetof(nb200_read_result, edits) == 24 && offsetof(nb200_read_result, status) == 28 &&
                  offsetof(nb200_read_result, reason) == 32 && offsetof(nb200_read_result, pair_score) == 36,
                  "the word-wise stores follow the layout of nb200_read_result");
    auto c16 = [](uint32_t v) { return v > 65535u ? 65535u : v; };
    rec[0] = (uint32_t)sc[0] | ((uint32_t)sc[1] << 16); rec[1] = (uint32_t)sc[2] | ((uint32_t)sc[3] << 16);
    rec[2] = nh[0] | (nh[1] << 16); rec[3] = nh[2] | (nh[3] << 16);
    rec[4] = c16(nc[0]) | (c16(nc[1]) << 16); rec[5] = c16(nc[2]) | (c16(nc[3]) << 16);
    rec[6] = (uint32_t)ed[0] | ((uint32_t)ed[1] << 8) | ((uint32_t)ed[2] << 16) | ((uint32_t)ed[3] << 24); rec[7] = (uint32_t)st[0] | ((uint32_t)st[1] << 8) | ((uint32_t)st[2] << 16) | ((uint32_t)st[3] << 24);
    rec[8] = (uint32_t)reason | ((uint32_t)(chosen < 0 ? 255 : chosen) << 8) | ((uint32_t)n_feat << 16) | (n_sw << 24);
    rec[9] = chosen < 0 ? 0u : chosen_score;
    return n_feat;
}

constexpr int kFastThreads = 256;      // call_fast_kernel block: one pair of same-address atomics per BLOCK for the two work lists
template <int NM>
__global__ void __launch_bounds__(kFastThreads)
call_fast_kernel(LibDev lib, CallParams cp, const OriSum *__restrict__ sums, uint32_t n_reads, uint32_t *__restrict__ slow_list,
                 uint32_t *__restrict__ setup_list, nb200_read_result *__restrict__ results, int32_t *__restrict__ feats,
                 uint16_t *__restrict__ row_nf, Counters *__restrict__ ctr) {
    constexpr int n_ro = NM * 2;
    constexpr bool paired = NM == 2;
    const uint32_t gw = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    bool active = gw < n_reads, slow = false, inmem = false;
    uint4 lo[n_ro], hi[n_ro];
    if (active) {
        const uint4 *src = reinterpret_cast<const uint4 *>(sums + (size_t)gw * n_ro);
#pragma unroll
        for (int q = 0; q < n_ro; q++) { lo[q] = __ldg(src + 2 * q); hi[q] = __ldg(src + 2 * q + 1); }
        if ((lo[0].y >> 8) & kSumWide) active = false;               // wide_kernel writes this read
    }
    uint32_t nh[4] = {0, 0, 0, 0}, nc[4] = {0, 0, 0, 0};
    int len[4] = {0, 0, 0, 0};
    if (active) {
#pragma unroll
        for (int q = 0; q < n_ro; q++) {
            nh[q] = lo[q].x & 0xFFFFu; len[q] = (int)(lo[q].y >> 16);
            const uint32_t flags = (lo[q].y >> 8) & 0xFFu;
            const int na = (int)(lo[q].y & 0xFFu);
            if (flags & kSumInMem) { slow = true; inmem = true; continue; }
            uint32_t c = 0;
            if (na > 0) c = __popc(hi[q].x) + (na > 1 ? __popc(hi[q].y) : 0) + (na > 2 ? __popc(hi[q].z) : 0) + (na > 3 ? __popc(hi[q].w) : 0);
            nc[q] = c;
            if (nh[q] && c && !(flags & kSumFull)) slow = true;      // partial hit: Smith-Waterman decides
        }
    }
    // reads that need Smith-Waterman and carry their candidate sets inline go to sw_setup_kernel (one THREAD per read);
    // reads with a candidate set in memory (more than 4 sparse words) to call_slow_kernel (one warp per read).
    // One atomic per warp and list.
    const bool setup = slow && !inmem;
    slow = slow && inmem;
    __shared__ uint32_t s_cnt[2][kFastThreads / 32];
    unsigned sb = 0, ub = 0;
    uint32_t my_base = 0;
    {
        // positions in the two lists: counts per warp -> one atomic per block and list (the returning atomics on one
        // address were 60 % of this kernel's stall samples when every warp issued its own)
        sb = __ballot_sync(kFull, active && slow); ub = __ballot_sync(kFull, active && setup);
        if (lane == 0) { s_cnt[0][threadIdx.x >> 5] = __popc(sb); s_cnt[1][threadIdx.x >> 5] = __popc(ub); }
        __syncthreads();
        if (threadIdx.x < 2) {          // issued now, consumed after the calling work below: the round trip of the atomic hides behind it
            uint32_t tot = 0;
#pragma unroll
            for (int w = 0; w < kFastThreads / 32; w++) tot += s_cnt[threadIdx.x][w];
            my_base = tot ? (uint32_t)atomicAdd(threadIdx.x ? &ctr->n_setup : &ctr->n_slow, (unsigned long long)tot) : 0u;
        }
    }
    slow = slow || setup;
    // Per-read outputs are staged in shared memory and written by the whole warp: a thread's own 40 B record and
    // max_hits feature ids would be 4- and 8-byte stores 40 B apart (32 sectors per instruction), the warp's 32 records are
    // one contiguous block.  Reads listed as slow, wide reads and the tail of the batch are left alone.
    extern __shared__ uint32_t stage[];
    const int mh = cp.max_hits;
    const int wib = threadIdx.x >> 5;
    uint32_t *s_res = stage + (size_t)wib * 32 * (10 + mh), *s_feat = s_res + 32 * 10;
    const bool mine = active && !slow;
    const unsigned okmask = __ballot_sync(kFull, mine);
    int n_feat = 0;
    if (mine) {
        int vbest[4];
#pragma unroll
        for (int o = 0; o < 4; o++) vbest[o] = nc[o] ? len[o] * kVW : -1;         // a hit orientation matched at every position here
        n_feat = thread_call<NM>(lib, cp, lo, hi, nh, nc, len, vbest, 0u, reinterpret_cast<int32_t *>(s_feat) + lane * mh, s_res + lane * 10);
        row_nf[gw] = (uint16_t)n_feat;
    }   // mine
    __syncwarp();
    const uint32_t gw0 = gw - (uint32_t)lane;                       // first read of this warp
    if (okmask) {
        uint2 *dst = reinterpret_cast<uint2 *>(results + gw0);      // 40 B records: five 8-byte words each
        const uint2 *src = reinterpret_cast<const uint2 *>(s_res);
        for (int t = lane; t < 32 * 5; t += 32)
            if ((okmask >> (t / 5)) & 1u) dst[t] = src[t];
        int32_t *fd = feats + (size_t)gw0 * mh;
        for (int t = lane; t < 32 * mh; t += 32)
            if ((okmask >> (t / mh)) & 1u) fd[t] = (int32_t)s_feat[t];
    }
    // the two work lists: block bases from the atomics issued above, then every listed read at base + its rank in the block
    {
        __shared__ uint32_t s_base[2];
        if (threadIdx.x < 2) s_base[threadIdx.x] = my_base;
        __syncthreads();
        const int wv = threadIdx.x >> 5;
        uint32_t b0 = s_base[0], b1 = s_base[1];
        for (int w = 0; w < wv; w++) { b0 += s_cnt[0][w]; b1 += s_cnt[1][w]; }
        if (active && slow && !setup) slow_list[b0 + __popc(sb & ((1u << lane) - 1))] = gw;
        if (active && setup) setup_list[b1 + __popc(ub & ((1u << lane) - 1))] = gw;
    }
}

// ---------------------------------------------------------------------------------------------
// Smith-Waterman setup, one THREAD per read (the reads call_fast_kernel listed in setup_list: at least one orientation
// hit partially, every candidate set has at most 4 sparse words and sits in the 32-byte summaries).  Per read: deferred
// slot + SW item range (one atomic per WARP hands out both for its 32 reads), orientation records, candidate sets parked
// for call_deferred_kernel, seed lookup, one work item per candidate in ascending reference order.  The work is a chain
// of dependent loads (summary -> record -> table bucket -> class record -> position), so it wants many reads in flight,
// not many lanes per read: a warp per read ran at 16 threads per instruction and 780 warp-instructions per read.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t rec_rank_thread(const LibDev &lib, const uint4 c_b, const uint4 c_w, uint32_t ref) {
    const uint32_t word = ref >> 5, below = (1u << (ref & 31)) - 1;
    if ((int32_t)c_w.z >= 0) {
        const uint32_t w0 = c_w.x & 0xFFFFu, w1 = c_w.x >> 16, w2 = c_w.y & 0xFFFFu, w3 = c_w.y >> 16;
        uint32_t rank = 0;
        rank += w0 < word ? __popc(c_b.x) : (w0 == word ? __popc(c_b.x & below) : 0);
        rank += w1 < word ? __popc(c_b.y) : (w1 == word ? __popc(c_b.y & below) : 0);
        rank += w2 < word ? __popc(c_b.z) : (w2 == word ? __popc(c_b.z & below) : 0);
        rank += w3 < word ? __popc(c_b.w) : (w3 == word ? __popc(c_b.w & below) : 0);
        return rank;
    }
    const int i = ov_find(lib, c_b.x, c_b.y, word);
    return __ldg(lib.ov_pre + c_b.x + i) + __popc(__ldg(lib.ov_b + c_b.x + i) & below);
}

template <int NM>
__global__ void __launch_bounds__(128)
sw_setup_kernel(LibDev lib, ReadsDev r1, ReadsDev r2, uint64_t read0, const OriSum *__restrict__ sums,
                const uint32_t *__restrict__ setup_list, RoRec *__restrict__ ro, uint32_t *__restrict__ roB,
                uint32_t *__restrict__ deferred, SwItem *__restrict__ items, uint32_t items_cap, Counters *__restrict__ ctr) {
    constexpr int n_ro = NM * 2;
    const int lane = threadIdx.x & 31;
    const uint32_t n_setup = (uint32_t)ctr->n_setup;
    const uint32_t stride = gridDim.x * blockDim.x;
    for (uint32_t d0 = (blockIdx.x * blockDim.x + threadIdx.x) & ~31u; d0 < n_setup; d0 += stride) {
        const uint32_t d = d0 + lane;
        const bool act = d < n_setup;
        const uint32_t gw = act ? setup_list[d] : 0u;
        uint4 lo[n_ro], hi[n_ro];
        uint32_t cnt[n_ro], n_items = 0;
        bool partial[n_ro];
#pragma unroll
        for (int q = 0; q < n_ro; q++) {
            cnt[q] = 0; partial[q] = false;
            lo[q] = make_uint4(0, 0, 0, 0); hi[q] = lo[q];
            if (!act) continue;
            const uint4 *src = reinterpret_cast<const uint4 *>(sums + (size_t)gw * n_ro + q);
            lo[q] = __ldg(src); hi[q] = __ldg(src + 1);
            const int na = (int)(lo[q].y & 0xFFu);
            const uint32_t flags = (lo[q].y >> 8) & 0xFFu, nh = lo[q].x & 0xFFFFu;
            uint32_t c = 0;
            if (nh && na > 0) c = __popc(hi[q].x) + (na > 1 ? __popc(hi[q].y) : 0) + (na > 2 ? __popc(hi[q].z) : 0) + (na > 3 ? __popc(hi[q].w) : 0);
            cnt[q] = c;
            partial[q] = c && !(flags & kSumFull);
            if (partial[q]) n_items += (c + 1) & ~1u;
        }
        // one atomic per warp: deferred slots and item ranges of its reads
        const unsigned ab = __ballot_sync(kFull, act);
        uint32_t wtot;
        const uint32_t ex = warp_excl_scan(n_items, lane, wtot);
        unsigned long long a = 0;
        if (lane == 0) a = atomicAdd(&ctr->alloc, ((unsigned long long)__popc(ab) << 40) | (unsigned long long)wtot);
        a = __shfl_sync(kFull, a, 0);
        if (!act) continue;
        const uint32_t dslot = (uint32_t)(a >> 40) + (uint32_t)__popc(ab & ((1u << lane) - 1));
        uint32_t off = (uint32_t)(a & kItemMask) + ex;
        const bool fits = (a & kItemMask) + ex + n_items <= items_cap;
        if (!fits) atomicAdd(&ctr->overflow, 1ull);
        deferred[dslot] = gw;
        const uint64_t read = read0 + gw;
#pragma unroll
        for (int q = 0; q < n_ro; q++) {
            const uint32_t ro_idx = dslot * n_ro + q;
            const int na = cnt[q] ? (int)(lo[q].y & 0xFFu) : 0;           // a set without members is an empty list
            const uint32_t len = lo[q].y >> 16;
            RoRec rr;
            rr.ncand = cnt[q]; rr.item_off = kInvalid; rr.n_hits = (uint16_t)(lo[q].x & 0xFFFFu); rr.len = (uint16_t)len;
            rr.na = (uint16_t)na; rr.full = (cnt[q] && !partial[q]) ? 1 : 0; rr.pad = 1;      // pad = 1: inline sets, finished by call_deferred_thread_kernel
            const uint32_t w[4] = {lo[q].z & 0xFFFFu, lo[q].z >> 16, lo[q].w & 0xFFFFu, lo[q].w >> 16};
            const uint32_t b[4] = {hi[q].x, hi[q].y, hi[q].z, hi[q].w};
            if (cnt[q]) {                                                  // park the class (read-indexed) for the deferred call
                uint32_t *dst = roB + ((size_t)gw * n_ro + q) * 2 * kCap;
#pragma unroll
                for (int j = 0; j < 4; j++) if (j < na) { dst[j] = w[j]; dst[kCap + j] = b[j]; }
            }
            if (partial[q]) {
                if (fits) {
                    rr.item_off = off;
                    const int seed_i = (int)(int16_t)(lo[q].x >> 16);
                    uint32_t seed_cls, seed_off;
                    seed_lookup(lib, q >= 2 ? r2 : r1, read, (int)len - lib.k + 1, q & 1, seed_i, seed_cls, seed_off);
                    uint4 s_b, s_w;
                    ldg256_cached(lib.class_rec + 2 * (size_t)seed_cls, s_b, s_w);
                    const uint32_t tag = ro_idx | (len << kRoIdxBits);
                    uint32_t at = off;
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        uint32_t bits = j < na ? b[j] : 0u;
                        while (bits) {
                            const uint32_t r = w[j] * 32 + (uint32_t)(__ffs(bits) - 1);
                            bits &= bits - 1;
                            const uint32_t pos = __ldg(lib.positions + seed_off + rec_rank_thread(lib, s_b, s_w, r));
                            SwItem it;
                            it.ro = tag; it.ref = r;
                            it.gwin = __ldg(lib.ref_gstart + r) + pos - (uint32_t)seed_i - (uint32_t)kBand;
                            it.v = 0;
                            items[at++] = it;
                        }
                    }
                    if (cnt[q] & 1) { SwItem it; it.ro = tag; it.ref = kInvalid; it.gwin = 0; it.v = 0; items[at] = it; }
                }
                off += (cnt[q] + 1) & ~1u;
            }
            ro[ro_idx] = rr;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// X4 for the reads call_fast_kernel listed, one warp per read: reads that need Smith-Waterman emit their work
// items, park their candidate sets and are finished by call_deferred_kernel after sw_kernel; reads with wide candidate
// sets but nothing to align are called here (call_read).
// ---------------------------------------------------------------------------------------------
template <int NM>
__global__ void __launch_bounds__(128)
call_slow_kernel(LibDev lib, CallParams cp, ReadsDev r1, ReadsDev r2, uint64_t read0, const OriSum *__restrict__ sums,
                 const uint32_t *__restrict__ slow_list, RoRec *__restrict__ ro, uint32_t *__restrict__ roB,
                 uint32_t *__restrict__ deferred, SwItem *__restrict__ items, uint32_t items_cap,
                 nb200_read_result *__restrict__ results, int32_t *__restrict__ feats, uint16_t *__restrict__ row_nf,
                 Counters *__restrict__ ctr) {
    __shared__ uint32_t smem[4 * kScratchWords];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    constexpr bool paired = NM == 2;
    constexpr int n_ro = NM * 2;
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    const uint32_t n_slow = (uint32_t)ctr->n_slow;
    List L4[4], T, Bst;
    carve_scratch(smem + (size_t)wib * kScratchWords, kCap, L4, T, Bst);
    for (uint32_t d = ((blockIdx.x * blockDim.x + threadIdx.x) >> 5); d < n_slow; d += warps) {
        const uint32_t gw = slow_list[d];
        const uint64_t read = read0 + gw;
        ReadState S;
        S.n_sw = 0;
        int seed_i[4];
        bool partial[4], in_mem[4];
        uint32_t n_items = 0;
        __syncwarp();
#pragma unroll
        for (int q = 0; q < 4; q++) {
            S.cls[q] = L4[q]; S.cls[q].n = 0;
            S.nc[q] = 0; S.nh[q] = 0; S.vbest[q] = -1; S.len[q] = 0; partial[q] = false; in_mem[q] = false; seed_i[q] = 0;
            if (q >= n_ro) continue;
            const uint4 *src = reinterpret_cast<const uint4 *>(sums + (size_t)gw * n_ro + q);
            const uint4 lo = __ldg(src), hi = __ldg(src + 1);
            const int na = (int)(lo.y & 0xFFu);
            const uint32_t flags = (lo.y >> 8) & 0xFFu;
            S.nh[q] = lo.x & 0xFFFFu; S.len[q] = (int)(lo.y >> 16);
            seed_i[q] = (int)(int16_t)(lo.x >> 16);
            in_mem[q] = (flags & kSumInMem) != 0;
            if (in_mem[q]) {
                const uint32_t *lst = roB + ((size_t)gw * n_ro + q) * 2 * kCap;
                for (int j = lane; j < na; j += 32) { L4[q].w[j] = lst[j]; L4[q].b[j] = lst[kCap + j]; }
            } else if (lane < na) {
                L4[q].w[lane] = lane == 0 ? (lo.z & 0xFFFFu) : (lane == 1 ? (lo.z >> 16) : (lane == 2 ? (lo.w & 0xFFFFu) : (lo.w >> 16)));
                L4[q].b[lane] = lane == 0 ? hi.x : (lane == 1 ? hi.y : (lane == 2 ? hi.z : hi.w));
            }
            L4[q].n = na;
            __syncwarp();
            const uint32_t cnt = S.nh[q] ? list_count(L4[q], lane) : 0u;
            if (!cnt) L4[q].n = 0;
            S.cls[q] = L4[q];
            S.nc[q] = cnt;
            const bool full = (flags & kSumFull) != 0;
            S.vbest[q] = cnt ? (full ? S.len[q] * kVW : 0) : -1;
            partial[q] = cnt && !full;
            if (partial[q]) n_items += (cnt + 1) & ~1u;
        }
        if (n_items == 0) {   // nothing to align: call the read now
            call_read(lib, cp, paired, S, T, Bst, lane, results + gw, feats + (size_t)gw * cp.max_hits, row_nf + gw, ctr);
            continue;
        }
        // ---- deferred: one atomic hands out the deferred slot and the SW item range -------------------
        unsigned long long a = 0;
        if (lane == 0) a = atomicAdd(&ctr->alloc, (1ull << 40) | (unsigned long long)n_items);
        a = __shfl_sync(kFull, a, 0);
        const uint32_t dslot = (uint32_t)(a >> 40);
        uint32_t off = (uint32_t)(a & kItemMask);
        const bool fits = (a & kItemMask) + n_items <= items_cap;
        if (!fits && lane == 0) atomicAdd(&ctr->overflow, 1ull);
        if (lane == 0) deferred[dslot] = gw;
#pragma unroll
        for (int q = 0; q < 4; q++) {
            if (q >= n_ro) continue;
            const uint32_t ro_idx = dslot * n_ro + q;
            RoRec rr;
            rr.ncand = S.nc[q]; rr.item_off = kInvalid; rr.n_hits = (uint16_t)S.nh[q]; rr.len = (uint16_t)S.len[q];
            rr.na = (uint16_t)S.cls[q].n; rr.full = (S.nc[q] && !partial[q]) ? 1 : 0; rr.pad = 0;
            if (S.nc[q] && !in_mem[q]) {            // park the class (read-indexed): the deferred call rebuilds B' on its words
                uint32_t *dst = roB + ((size_t)gw * n_ro + q) * 2 * kCap;
                for (int j = lane; j < S.cls[q].n; j += 32) { dst[j] = S.cls[q].w[j]; dst[kCap + j] = S.cls[q].b[j]; }
            }
            if (partial[q]) {
                if (fits) {
                    rr.item_off = off;
                    const ReadsDev &R = q >= 2 ? r2 : r1;
                    uint32_t seed_cls, seed_off;
                    seed_lookup(lib, R, read, S.len[q] - lib.k + 1, q & 1, seed_i[q], seed_cls, seed_off);
                    emit_items(lib, S.cls[q], seed_cls, seed_off, seed_i[q], ro_idx, (uint32_t)S.len[q], S.nc[q], items, off, lane);
                }
                off += (S.nc[q] + 1) & ~1u;
            }
            if (lane == 0) ro[ro_idx] = rr;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// X3c: banded Smith-Waterman, linear gap, two candidates of the same oriented read per thread
// in the two s16 halves of DPX s16x2 instructions (VIADDMNMX / VIMNMX3).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t spread_bits32(uint32_t v) {   // bit b -> bit 2b
    uint64_t x = v;
    x = (x | (x << 16)) & 0x0000FFFF0000FFFFull;
    x = (x | (x << 8)) & 0x00FF00FF00FF00FFull;
    x = (x | (x << 4)) & 0x0F0F0F0F0F0F0F0Full;
    x = (x | (x << 2)) & 0x3333333333333333ull;
    x = (x | (x << 1)) & 0x5555555555555555ull;
    return x;
}

__device__ __forceinline__ void load_ref_window(const LibDev &lib, uint32_t g, uint64_t &bases, uint64_t &nspread) {
    // 32 bases starting at global coordinate g
    const uint32_t w = g >> 5, sh = (g & 31) * 2;
    const uint64_t a = __ldg(lib.ref2bit + w), b = __ldg(lib.ref2bit + w + 1);
    bases = sh ? ((a >> sh) | (b << (64 - sh))) : a;
    const uint64_t n01 = (uint64_t)__ldg(lib.refN + w) | ((uint64_t)__ldg(lib.refN + w + 1) << 32);
    nspread = spread_bits32((uint32_t)(n01 >> (g & 31)));
}

// One 32-base reference window as 32-bit halves; shifted right by one base per DP row.
struct RefWin { uint32_t lo, hi, nlo, nhi; };

__device__ __forceinline__ void load_ref_window32(const LibDev &lib, uint32_t g, RefWin &w) {
    uint64_t bases, nspread;
    load_ref_window(lib, g, bases, nspread);
    w.lo = (uint32_t)bases; w.hi = (uint32_t)(bases >> 32);
    w.nlo = (uint32_t)nspread; w.nhi = (uint32_t)(nspread >> 32);
}
__device__ __forceinline__ void shift_ref_window(RefWin &w) {       // drop one base
    w.lo = __funnelshift_r(w.lo, w.hi, 2); w.hi >>= 2;
    w.nlo = __funnelshift_r(w.nlo, w.nhi, 2); w.nhi >>= 2;
}
// match bits of the 17 band cells of this row: bit 2b of lo for b < 16, bit 0 of hi for b = 16
__device__ __forceinline__ void row_matches(const RefWin &w, uint32_t qrep, uint32_t qmask, uint32_t &zlo, uint32_t &zhi) {
    const uint32_t ylo = w.lo ^ qrep, yhi = w.hi ^ qrep;
    zlo = ~(ylo | (ylo >> 1)) & ~w.nlo & 0x55555555u & qmask;
    zhi = ~(yhi | (yhi >> 1)) & ~w.nhi & 1u & qmask;
}

// One DP row of the band for two alignments at once (s16 halves).  y0/y1/y2: match flags of cells 0-7 / 8-15 / 16
// (cell b at bit 2(b & 7) of each half).  H = max(0, diag + s, max(up, left) + gap): packed add, packed max,
// DPX add-max with ReLU (VIADDMNMX.S16x2.RELU); row maxima with the DPX three-way max (VIMNMX3.S16x2).
// s16 headroom: a read that reaches SW has a k-mer the library lacks, so no window matches all of its bases; at 500
// bases V <= 64 * 499, and diag + kMatchDelta < 64 * 499 + 193 < 32767 (test_long_reads_gpu.py::test_sw_near_s16_ceiling).
__device__ __forceinline__ void sw_row(uint32_t (&H)[kNB], uint32_t y0, uint32_t y1, uint32_t y2, uint32_t &best) {
    uint32_t left = 0, rowmax = 0;
#pragma unroll
    for (int b = 0; b < kNB; b++) {
        const uint32_t y = b < 8 ? y0 : (b < 16 ? y1 : y2);
        const uint32_t mf = (y >> (2 * (b & 7))) & 0x00010001u;    // match flag per s16 half
        const uint32_t a = mf * kMatchDelta + H[b];                 // diag + (match - mismatch)
        const uint32_t up = (b + 1 < kNB) ? H[b + 1] : 0u;
        const uint32_t h = __viaddmax_s16x2_relu(__vmaxs2(up, left), kGP, __vadd2(a, kXP));
        H[b] = h;
        if (b & 1) rowmax = __vimax3_s16x2(rowmax, left, h); else if (b == kNB - 1) rowmax = __vimax3_s16x2(rowmax, h, h);
        left = h;
    }
    best = __vimax3_s16x2(best, rowmax, rowmax);
}

// best V of the oriented read against two candidates (low half: gA, high half: gB)
__device__ __forceinline__ uint32_t sw_pair(const LibDev &lib, const uint64_t *seq, const uint32_t *nm, int L, int ori,
                                            uint32_t gA, uint32_t gB) {
    uint32_t H[kNB];
#pragma unroll
    for (int b = 0; b < kNB; b++) H[b] = 0;
    uint32_t best = 0;
    RefWin wa, wb;
    wa.lo = wa.hi = wa.nlo = wa.nhi = 0; wb = wa;
    for (int i = 0; i < L; i++) {
        if ((i & 15) == 0) {               // one 32-base window serves 16 rows of 17 cells
            load_ref_window32(lib, gA + i, wa);
            load_ref_window32(lib, gB + i, wb);
        }
        const int idx = ori ? (L - 1 - i) : i;
        uint32_t q = (uint32_t)(seq[idx >> 5] >> (2 * (idx & 31))) & 3u;
        if (ori) q = 3u - q;
        const uint32_t qn = (nm[idx >> 5] >> (idx & 31)) & 1u;
        const uint32_t qrep = q * 0x55555555u;           // the base replicated over all 16 two-bit groups
        const uint32_t qmask = qn - 1u;                  // read N: no cell of the row matches
        uint32_t za_lo, za_hi, zb_lo, zb_hi;
        row_matches(wa, qrep, qmask, za_lo, za_hi);
        row_matches(wb, qrep, qmask, zb_lo, zb_hi);
        shift_ref_window(wa);
        shift_ref_window(wb);
        // pack A (low s16 half) and B (high half): cell b of y0 at bits 2b / 16+2b, b < 8; y1: cells 8..15
        const uint32_t y0 = __byte_perm(za_lo, zb_lo, 0x5410);
        const uint32_t y1 = __byte_perm(za_lo, zb_lo, 0x7632);
        const uint32_t y2 = za_hi | (zb_hi << 16);
        sw_row(H, y0, y1, y2, best);
    }
    return best;
}

// ---------------------------------------------------------------------------------------------
// Candidates of one oriented read are alleles that agree on every k-mer the read hit, so most of
// their band windows (L + 16 reference bases from gwin) are IDENTICAL and so are their V.
// Two thread-per-item passes: window_hash_kernel fingerprints every candidate's window;
// dedupe_kernel looks back over the (contiguous) items of the same read orientation for the first
// one with the same fingerprint, VERIFIES the two windows word by word, and either records it as
// its representative or appends the item to the flat work list of sw_kernel.  The look-back is
// bounded (kLookBack items), so a representative may itself have one: readers follow rep[] to
// the root.  Nothing is modified in place, so the passes need no ordering between threads.
// ---------------------------------------------------------------------------------------------
constexpr int kLookBack = 32;

__device__ __forceinline__ void window_word(const LibDev &lib, uint32_t g, int w, int rem_last, int n_w, uint64_t &bases, uint32_t &nbits) {
    const uint32_t gg = g + 32u * (uint32_t)w;
    const uint32_t wi = gg >> 5, sh = (gg & 31) * 2;
    const uint64_t a = __ldg(lib.ref2bit + wi), b = __ldg(lib.ref2bit + wi + 1);
    bases = sh ? ((a >> sh) | (b << (64 - sh))) : a;
    const uint64_t n01 = (uint64_t)__ldg(lib.refN + wi) | ((uint64_t)__ldg(lib.refN + wi + 1) << 32);
    nbits = (uint32_t)(n01 >> (gg & 31));
    if (w == n_w - 1 && rem_last < 32) { bases &= (1ull << (2 * rem_last)) - 1; nbits &= (1u << rem_last) - 1; }
}

__global__ void __launch_bounds__(256)
window_hash_kernel(LibDev lib, SwItem *__restrict__ items, uint32_t items_cap, const Counters *__restrict__ ctr) {
    const unsigned long long total = ctr->alloc & kItemMask;
    if (total > items_cap) return;
    for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < (uint32_t)total; t += gridDim.x * blockDim.x) {
        const SwItem it = items[t];
        if (it.ref == kInvalid) continue;                  // padding of an odd segment
        const int W = (int)((it.ro >> kRoIdxBits) & 0x1FF) + 2 * kBand;
        const int n_w = (W + 31) >> 5, rem_last = W - 32 * (n_w - 1);
        uint64_t h = 0x9E3779B97F4A7C15ull;
        if (n_w <= 6) {                                    // reads <= 176 bases: all loads in flight before the first use
            uint64_t bs[6]; uint32_t nb[6];
#pragma unroll
            for (int w = 0; w < 6; w++) { bs[w] = 0; nb[w] = 0; if (w < n_w) window_word(lib, it.gwin, w, rem_last, n_w, bs[w], nb[w]); }
#pragma unroll
            for (int w = 0; w < 6; w++)
                if (w < n_w) {
                    h = (h ^ bs[w]) * 0xD6E8FEB86659FD93ull;
                    h = (h ^ (h >> 32) ^ nb[w]) * 0x9FB21C651E98DF25ull;
                }
        } else {
            for (int w = 0; w < n_w; w++) {
                uint64_t bs; uint32_t nb;
                window_word(lib, it.gwin, w, rem_last, n_w, bs, nb);
                h = (h ^ bs) * 0xD6E8FEB86659FD93ull;
                h = (h ^ (h >> 32) ^ nb) * 0x9FB21C651E98DF25ull;
            }
        }
        items[t].v = (uint32_t)(h >> 32) ^ (uint32_t)h;      // overwritten by the score for the items that get aligned
    }
}

__global__ void __launch_bounds__(256)
dedupe_kernel(LibDev lib, const SwItem *__restrict__ items, uint32_t items_cap, uint32_t *__restrict__ rep,
              uint32_t *__restrict__ uniq, Counters *__restrict__ ctr) {
    const unsigned long long total = ctr->alloc & kItemMask;
    if (total > items_cap) return;
    const int lane = threadIdx.x & 31;
    const uint32_t n = (uint32_t)total;
    uint32_t dups = 0;
    for (uint32_t t0 = (blockIdx.x * blockDim.x + threadIdx.x) & ~31u; t0 < n; t0 += gridDim.x * blockDim.x) {
        const uint32_t t = t0 + lane;
        SwItem it;
        it.ro = 0; it.ref = kInvalid; it.gwin = 0; it.v = 0;
        if (t < n) it = items[t];
        const bool live = it.ref != kInvalid;
        uint32_t r = t;
        if (live) {
            const int W = (int)((it.ro >> kRoIdxBits) & 0x1FF) + 2 * kBand;
            const int n_w = (W + 31) >> 5, rem_last = W - 32 * (n_w - 1);
            const uint32_t seg = it.ro & kRoIdxMask;
            // earliest item of the same segment within the look-back with the same fingerprint ...
            uint32_t e = t;
            for (int back = 1; back <= kLookBack && back <= (int)t; back++) {
                const uint32_t oro = items[t - back].ro, ov = items[t - back].v;
                if ((oro & kRoIdxMask) != seg) break;
                if (ov == it.v) e = t - back;
            }
            if (e != t) {                                  // ... and a fingerprint is not a proof: compare the windows
                const uint32_t og = items[e].gwin;
                bool same = true;
                for (int w = 0; w < n_w && same; w++) {
                    uint64_t b0, b1; uint32_t n0, n1;
                    window_word(lib, it.gwin, w, rem_last, n_w, b0, n0);
                    window_word(lib, og, w, rem_last, n_w, b1, n1);
                    same = (b0 == b1) && (n0 == n1);
                }
                if (same) r = e;
            }
            rep[t] = r;
        }
        const bool uq = live && r == t;
        const unsigned ub = __ballot_sync(kFull, uq);
        if (ub) {
            uint32_t base = 0;
            if (lane == 0) base = (uint32_t)atomicAdd(&ctr->n_swpairs, (unsigned long long)__popc(ub));
            base = __shfl_sync(kFull, base, 0);
            if (uq) uniq[base + __popc(ub & ((1u << lane) - 1))] = t;
        }
        dups += (live && !uq) ? 1u : 0u;
    }
    dups = warp_sum(dups);
    if (lane == 0 && dups) atomicAdd(&ctr->sw_dups, (unsigned long long)dups);
}

// best V of two (oriented read, window) items, one per s16 half; the two may belong to different reads
struct SwQuery {
    const uint64_t *seq;
    const uint32_t *nm;
    int L, ori;
};
__device__ __forceinline__ void query_base(const SwQuery &q, int i, uint32_t &qrep, uint32_t &qmask) {
    const bool in = i < q.L;
    const int idx = in ? (q.ori ? (q.L - 1 - i) : i) : 0;
    uint32_t b = (uint32_t)(q.seq[idx >> 5] >> (2 * (idx & 31))) & 3u;
    if (q.ori) b = 3u - b;
    const uint32_t qn = (q.nm[idx >> 5] >> (idx & 31)) & 1u;
    qrep = b * 0x55555555u;
    qmask = in ? (qn - 1u) : 0u;                           // read N or past the end of the shorter read: no cell matches
}
__device__ __forceinline__ uint32_t sw_pair2(const LibDev &lib, const SwQuery &qa, const SwQuery &qb, uint32_t gA, uint32_t gB) {
    uint32_t H[kNB];
#pragma unroll
    for (int b = 0; b < kNB; b++) H[b] = 0;
    uint32_t best = 0;
    RefWin wa, wb;
    wa.lo = wa.hi = wa.nlo = wa.nhi = 0; wb = wa;
    const int Lmax = max(qa.L, qb.L);
    for (int i = 0; i < Lmax; i++) {
        if ((i & 15) == 0) {
            load_ref_window32(lib, gA + i, wa);
            load_ref_window32(lib, gB + i, wb);
        }
        uint32_t qrepA, qmaskA, qrepB, qmaskB;
        query_base(qa, i, qrepA, qmaskA);
        query_base(qb, i, qrepB, qmaskB);
        uint32_t za_lo, za_hi, zb_lo, zb_hi;
        row_matches(wa, qrepA, qmaskA, za_lo, za_hi);
        row_matches(wb, qrepB, qmaskB, zb_lo, zb_hi);
        shift_ref_window(wa);
        shift_ref_window(wb);
        const uint32_t y0 = __byte_perm(za_lo, zb_lo, 0x5410);
        const uint32_t y1 = __byte_perm(za_lo, zb_lo, 0x7632);
        const uint32_t y2 = za_hi | (zb_hi << 16);
        sw_row(H, y0, y1, y2, best);
    }
    return best;
}

__global__ void __launch_bounds__(128)
sw_kernel(LibDev lib, ReadsDev r1, ReadsDev r2, uint64_t read0, int n_mates, const uint32_t *__restrict__ deferred,
          SwItem *__restrict__ items, uint32_t items_cap, const uint32_t *__restrict__ uniq, Counters *__restrict__ ctr) {
    if ((ctr->alloc & kItemMask) > items_cap) return;     // overflowed batch: nothing valid, the host retries
    const uint32_t n_items = (uint32_t)ctr->n_swpairs;    // distinct windows listed by dedupe_kernel
    const uint32_t n_thr = (n_items + 1) >> 1;
    const int n_ro = n_mates * 2;
    unsigned long long my_cells = 0, my_pairs = 0;
    for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < n_thr; t += gridDim.x * blockDim.x) {
        const uint32_t ua = uniq[2 * t];
        const bool hasB = 2 * t + 1 < n_items;
        const uint32_t ub = hasB ? uniq[2 * t + 1] : ua;
        const SwItem ia = items[ua], ib = items[ub];
        SwQuery q[2];
#pragma unroll
        for (int hlf = 0; hlf < 2; hlf++) {
            const uint32_t roi = (hlf ? ib.ro : ia.ro) & kRoIdxMask;
            const uint32_t sub = roi % n_ro;
            const uint64_t read = read0 + deferred[roi / n_ro];
            const ReadsDev R = (sub >> 1) ? r2 : r1;
            const uint8_t *rec = R.packed + read * R.stride;
            q[hlf].seq = reinterpret_cast<const uint64_t *>(rec);
            q[hlf].nm = reinterpret_cast<const uint32_t *>(rec + (size_t)R.words * 8);
            q[hlf].L = read_length(R, read);
            q[hlf].ori = (int)(sub & 1);
        }
        const uint32_t best = sw_pair2(lib, q[0], q[1], ia.gwin, ib.gwin);
        items[ua].v = best & 0xFFFFu;
        if (hasB) items[ub].v = best >> 16;
        my_pairs += hasB ? 2 : 1;
        my_cells += ((unsigned long long)q[0].L + (hasB ? (unsigned long long)q[1].L : 0ull)) * kNB;
    }
    // one atomic per warp
    for (int o = 16; o; o >>= 1) {
        my_cells += __shfl_xor_sync(kFull, my_cells, o);
        my_pairs += __shfl_xor_sync(kFull, my_pairs, o);
    }
    if ((threadIdx.x & 31) == 0 && my_pairs) {
        atomicAdd(&ctr->sw_cells, my_cells);
        atomicAdd(&ctr->sw_pairs, my_pairs);
    }
}

// ---------------------------------------------------------------------------------------------
// Deferred X4, one THREAD per read that went through Smith-Waterman with inline candidate sets (RoRec.pad = 1, written
// by sw_setup_kernel): best V over the candidates (each candidate's score is the score of the root of its
// representative chain, dedupe_kernel), refinement B' = {V >= V* - 193 num_mismatches}, then thread_call.
// Like the setup, this is a chain of dependent loads per read (record -> item -> representative -> score): many reads
// in flight beat many lanes per read.
// ---------------------------------------------------------------------------------------------
template <int NM>
__global__ void __launch_bounds__(128)
call_deferred_thread_kernel(LibDev lib, CallParams cp, const RoRec *__restrict__ ro, const uint32_t *__restrict__ roB,
                            const uint32_t *__restrict__ deferred, const SwItem *__restrict__ items, const uint32_t *__restrict__ rep,
                            uint32_t items_cap, nb200_read_result *__restrict__ results, int32_t *__restrict__ feats,
                            uint16_t *__restrict__ row_nf, uint32_t *__restrict__ warp_list, Counters *__restrict__ ctr) {
    const unsigned long long alloc = ctr->alloc;
    if ((alloc & kItemMask) > items_cap) return;         // overflowed batch: the host retries
    const uint32_t n_def = (uint32_t)(alloc >> 40);
    constexpr int n_ro = NM * 2;
    const int mh = cp.max_hits;
    for (uint32_t d = blockIdx.x * blockDim.x + threadIdx.x; d < n_def; d += gridDim.x * blockDim.x) {
        RoRec rr[n_ro];
#pragma unroll
        for (int o = 0; o < n_ro; o++) rr[o] = ro[(size_t)d * n_ro + o];
        if (!rr[0].pad) { warp_list[atomicAdd(&ctr->n_warpdef, 1ull)] = d; continue; }     // candidate sets in memory (rare): listed for the warp-per-read kernel
        const uint32_t gw = deferred[d];
        uint4 lo[n_ro], hi[n_ro];
        uint32_t nh[4] = {0, 0, 0, 0}, nc[4] = {0, 0, 0, 0}, n_sw = 0;
        int len[4] = {0, 0, 0, 0}, vbest[4] = {-1, -1, -1, -1};
#pragma unroll
        for (int o = 0; o < n_ro; o++) {
            nh[o] = rr[o].n_hits; len[o] = rr[o].len;
            lo[o] = make_uint4(0u, 0u, 0xFFFFFFFFu, 0xFFFFFFFFu); hi[o] = make_uint4(0u, 0u, 0u, 0u);
            if (rr[o].n_hits == 0 || rr[o].ncand == 0) continue;
            const uint32_t *src = roB + ((size_t)gw * n_ro + o) * 2 * kCap;        // candidate sets are parked by read
            const int na = rr[o].na;
            uint32_t w[4] = {0xFFFFu, 0xFFFFu, 0xFFFFu, 0xFFFFu}, b[4] = {0u, 0u, 0u, 0u};
#pragma unroll
            for (int j = 0; j < 4; j++) if (j < na) { w[j] = src[j]; if (rr[o].full) b[j] = src[kCap + j]; }
            if (rr[o].full) {
                vbest[o] = (int)rr[o].len * kVW;
                nc[o] = rr[o].ncand;
            } else {
                n_sw++;
                const uint32_t i0 = rr[o].item_off, ncand = rr[o].ncand;
                auto item_v = [&](uint32_t t) -> uint32_t {
                    uint32_t a = i0 + t, r = rep[a];
                    while (r != a) { a = r; r = rep[a]; }
                    return items[a].v;
                };
                // the first 8 candidates (nearly always all of them): scores and references fetched by an unrolled loop, so
                // that the dependent loads rep -> item of different candidates are in flight together, and kept for pass 2
                uint32_t vv[8], rf[8];
                uint32_t vb = 0;
#pragma unroll
                for (int t = 0; t < 8; t++) {
                    vv[t] = 0; rf[t] = 0;
                    if ((uint32_t)t < ncand) { vv[t] = item_v((uint32_t)t); rf[t] = items[i0 + t].ref; vb = max(vb, vv[t]); }
                }
                for (uint32_t t = 8; t < ncand; t++) vb = max(vb, item_v(t));
                const uint32_t slack = (uint32_t)cp.num_mismatches * kMatchDelta;
                const uint32_t vmin = vb > slack ? vb - slack : 0u;
                uint32_t c = 0;
                auto keep = [&](uint32_t ref) {
                    const uint32_t word = ref >> 5, bit = 1u << (ref & 31);
#pragma unroll
                    for (int j = 0; j < 4; j++) if (w[j] == word) b[j] |= bit;
                    c++;
                };
#pragma unroll
                for (int t = 0; t < 8; t++) if ((uint32_t)t < ncand && vv[t] >= vmin) keep(rf[t]);
                for (uint32_t t = 8; t < ncand; t++) if (item_v(t) >= vmin) keep(items[i0 + t].ref);
                nc[o] = c;
                vbest[o] = (int)vb;
            }
            lo[o] = make_uint4(0u, (uint32_t)na, w[0] | (w[1] << 16), w[2] | (w[3] << 16));
            hi[o] = make_uint4(b[0], b[1], b[2], b[3]);
        }
        uint32_t rec[10];
        int32_t *fout = feats + (uint64_t)gw * mh;
        const int n_feat = thread_call<NM>(lib, cp, lo, hi, nh, nc, len, vbest, n_sw, fout, rec);
        uint2 *dst = reinterpret_cast<uint2 *>(results + gw);        // 40 B records, 8-byte aligned
#pragma unroll
        for (int t = 0; t < 5; t++) dst[t] = make_uint2(rec[2 * t], rec[2 * t + 1]);
        row_nf[gw] = (uint16_t)n_feat;
    }
}

// ---------------------------------------------------------------------------------------------
// Deferred X4: reads that went through Smith-Waterman.  One warp per deferred read.
// ---------------------------------------------------------------------------------------------
template <int NM>
__global__ void __launch_bounds__(256)
call_deferred_kernel(LibDev lib, CallParams cp, const RoRec *__restrict__ ro,
                     const uint32_t *__restrict__ roB, const uint32_t *__restrict__ deferred,
                     const SwItem *__restrict__ items, const uint32_t *__restrict__ rep, uint32_t items_cap,
                     nb200_read_result *__restrict__ results, int32_t *__restrict__ feats,
                     uint16_t *__restrict__ row_nf, const uint32_t *__restrict__ warp_list, Counters *__restrict__ ctr) {
    __shared__ uint32_t smem[8 * kScratchWords];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const unsigned long long alloc = ctr->alloc;
    if ((alloc & kItemMask) > items_cap) return;         // overflowed batch: the host retries
    const uint32_t n_def = (uint32_t)(alloc >> 40);
    constexpr int n_ro = NM * 2;
    constexpr bool paired = NM == 2;
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    List L4[4], T, Bst;
    carve_scratch(smem + (size_t)wib * kScratchWords, kCap, L4, T, Bst);
    (void)n_def;
    const uint32_t n_list = (uint32_t)ctr->n_warpdef;    // the deferred reads call_deferred_thread_kernel left for this kernel
    for (uint32_t t = ((blockIdx.x * blockDim.x + threadIdx.x) >> 5); t < n_list; t += warps) {
        const uint32_t d = warp_list[t];
        const uint32_t gw = deferred[d];
        ReadState S;
        S.n_sw = 0;
        __syncwarp();
#pragma unroll
        for (int o = 0; o < 4; o++) {
            S.cls[o] = L4[o]; S.cls[o].n = 0;
            S.nc[o] = 0; S.nh[o] = 0; S.vbest[o] = -1; S.len[o] = 0;
            if (o >= n_ro) continue;
            const uint32_t ro_idx = d * n_ro + o;
            const RoRec rr = ro[ro_idx];
            S.nh[o] = rr.n_hits; S.len[o] = rr.len;
            if (rr.n_hits == 0 || rr.ncand == 0) continue;
            const uint32_t *src = roB + ((size_t)gw * n_ro + o) * 2 * kCap;        // candidate sets are parked by read
            const bool keep_bits = rr.full != 0;
            for (int j = lane; j < (int)rr.na; j += 32) { L4[o].w[j] = src[j]; L4[o].b[j] = keep_bits ? src[kCap + j] : 0u; }
            S.cls[o].n = rr.na;
            __syncwarp();
            if (rr.full) {
                S.vbest[o] = (int)rr.len * kVW;
                S.nc[o] = rr.ncand;
            } else {
                S.n_sw++;
                const SwItem *seg = items + rr.item_off;
                uint32_t vb = 0;
                // the score of a candidate is the score of the root of its representative chain (dedupe_kernel)
                auto item_v = [&](uint32_t t) -> uint32_t {
                    uint32_t a = rr.item_off + t, b = rep[a];
                    while (b != a) { a = b; b = rep[a]; }
                    return items[a].v;
                };
                for (uint32_t t = lane; t < rr.ncand; t += 32) vb = max(vb, item_v(t));
                const uint32_t vbest = warp_max(vb);
                const uint32_t slack = (uint32_t)cp.num_mismatches * kMatchDelta;
                const uint32_t vmin = vbest > slack ? vbest - slack : 0u;
                for (uint32_t t = lane; t < rr.ncand; t += 32) {
                    const SwItem it = seg[t];
                    const uint32_t v = item_v(t);
                    if (v >= vmin) atomicOr(&L4[o].b[list_find(S.cls[o], it.ref >> 5)], 1u << (it.ref & 31));
                }
                __syncwarp();
                S.nc[o] = list_count(S.cls[o], lane);
                S.vbest[o] = (int)vbest;
            }
        }
        call_read(lib, cp, paired, S, T, Bst, lane, results + gw, feats + (uint64_t)gw * cp.max_hits, row_nf + gw, ctr);
    }
}

// ---------------------------------------------------------------------------------------------
// Wide reads (narrowest class spans more than kCap reference words): same device functions on
// global scratch sized for the whole library, Smith-Waterman done by the lanes of the warp.
// Rare by construction; correctness over speed.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
wide_kernel(LibDev lib, CallParams cp, ReadsDev r1, ReadsDev r2, uint64_t read0, int n_mates,
            const uint32_t *__restrict__ wide_list, uint32_t *__restrict__ scratch, uint32_t *__restrict__ vbuf,
            nb200_read_result *__restrict__ results, int32_t *__restrict__ feats, uint16_t *__restrict__ row_nf,
            Counters *__restrict__ ctr) {
    const int lane = threadIdx.x & 31;
    const uint32_t wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    const uint32_t n_wide = (uint32_t)ctr->n_wide;
    const uint32_t cap = lib.n_words;
    const bool paired = n_mates == 2;
    List L4[4], T, Bst;
    carve_scratch(scratch + (size_t)wid * 16 * cap, cap, L4, T, Bst);
    uint32_t *V = vbuf + (size_t)wid * ((size_t)lib.n_words * 32 + 32);
    for (uint32_t t = wid; t < n_wide; t += warps) {
        const uint32_t gw = wide_list[t];
        const uint64_t read = read0 + gw;
        ReadState S;
        S.n_sw = 0;
        uint32_t n_probe = 0, slots = 0;
        __syncwarp();
#pragma unroll
        for (int m = 0; m < 2; m++) {
            if (m >= n_mates) {
#pragma unroll
                for (int o = 0; o < 2; o++) { const int q = m * 2 + o; S.cls[q] = L4[q]; S.cls[q].n = 0; S.nc[q] = 0; S.nh[q] = 0; S.vbest[q] = -1; S.len[q] = 0; }
                continue;
            }
            const ReadsDev R = m ? r2 : r1;
            MateProbe M;
            probe_mate<false>(lib, R, read, lane, cap, &L4[m * 2], M, n_probe, slots);
            owner_to_list(M, &L4[m * 2], lane);
            const uint8_t *rec = R.packed + read * R.stride;
            const uint64_t *seq = reinterpret_cast<const uint64_t *>(rec);
            const uint32_t *nm = reinterpret_cast<const uint32_t *>(rec + (size_t)R.words * 8);
#pragma unroll
            for (int o = 0; o < 2; o++) {
                const int q = m * 2 + o;
                __syncwarp();
                uint32_t cnt = M.nh[o] ? list_count(L4[q], lane) : 0u;
                if (!cnt) L4[q].n = 0;
                S.cls[q] = L4[q];
                S.nh[q] = M.nh[o]; S.len[q] = M.L; S.nc[q] = cnt;
                const bool full = M.nh[o] && (int)M.nh[o] == M.P;
                S.vbest[q] = cnt ? (full ? M.L * kVW : 0) : -1;
                if (cnt && !full) {
                    // candidates (ascending) -> V by the lanes, two per call in the s16 halves
                    S.n_sw++;
                    uint32_t seed_cls, seed_off;
                    seed_lookup(lib, R, read, M.P, o, M.seed_i[o], seed_cls, seed_off);
                    const Rec seed = load_rec(lib, seed_cls);
                    uint32_t run = 0;
                    for (int base = 0; base < L4[q].n; base += 32) {        // 1. list the candidates' windows in V
                        const int j = base + lane;
                        uint32_t bits = j < L4[q].n ? L4[q].b[j] : 0u, tot;
                        uint32_t ex = run + warp_excl_scan(__popc(bits), lane, tot);
                        while (bits) {
                            const int b = __ffs(bits) - 1;
                            bits &= bits - 1;
                            const uint32_t r = L4[q].w[j] * 32 + b;
                            const uint32_t pos = __ldg(lib.positions + seed_off + rec_rank(lib, seed, r));
                            V[ex++] = __ldg(lib.ref_gstart + r) + pos - (uint32_t)M.seed_i[o] - (uint32_t)kBand;
                        }
                        run += tot;
                    }
                    __syncwarp();
                    uint32_t vb = 0;
                    for (uint32_t c0 = 2 * lane; c0 < cnt; c0 += 64) {      // 2. align
                        const uint32_t gA = V[c0], gB = (c0 + 1 < cnt) ? V[c0 + 1] : gA;
                        const uint32_t best = sw_pair(lib, seq, nm, M.L, o, gA, gB);
                        V[c0] = best & 0xFFFFu;
                        vb = max(vb, best & 0xFFFFu);
                        if (c0 + 1 < cnt) { V[c0 + 1] = best >> 16; vb = max(vb, best >> 16); }
                    }
                    __syncwarp();
                    const uint32_t vbest = warp_max(vb);
                    const uint32_t slack = (uint32_t)cp.num_mismatches * kMatchDelta;
                    const uint32_t vmin = vbest > slack ? vbest - slack : 0u;
                    run = 0;
                    for (int base = 0; base < L4[q].n; base += 32) {        // 3. keep the survivors
                        const int j = base + lane;
                        const uint32_t bits0 = j < L4[q].n ? L4[q].b[j] : 0u;
                        uint32_t bits = bits0, keep = 0, tot;
                        uint32_t ex = run + warp_excl_scan(__popc(bits), lane, tot);
                        while (bits) {
                            const int b = __ffs(bits) - 1;
                            bits &= bits - 1;
                            if (V[ex++] >= vmin) keep |= 1u << b;
                        }
                        if (j < L4[q].n) L4[q].b[j] = keep;
                        run += tot;
                    }
                    __syncwarp();
                    S.nc[q] = list_count(L4[q], lane);
                    S.vbest[q] = (int)vbest;
                    if (lane == 0) { atomicAdd(&ctr->sw_pairs, (unsigned long long)cnt); atomicAdd(&ctr->sw_cells, (unsigned long long)cnt * M.L * kNB); }
                }
            }
        }
        __syncwarp();
        call_read(lib, cp, paired, S, T, Bst, lane, results + gw, feats + (uint64_t)gw * cp.max_hits, row_nf + gw, ctr);
    }
}

}  // namespace nb200
