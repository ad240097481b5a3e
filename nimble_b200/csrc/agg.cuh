// A6 on device: (cell, umi, feature list, score) rows -> per-cell UMI counts
// (reference nimble/__main__.py:234-293 + nimble/utils.py:119-224; pinned by oracle/ + tests/golden).
//
// Ordering trick: pandas sorts rows by the comma-joined feature STRING; lexicographic order of
// per-position token ranks (name+',' inner / name+NUL last) reproduces that byte order exactly, so no
// string is ever compared on the device.
//
// Stage 1: rows -> stable radix sort by the 64-bit (cell, umi) key -> rows of a UMI into feature-string order
// (per-group insertion sort) -> umi_simple_kernel settles the UMIs whose rows all carry one list (most of them) and
// lists the others for umi_general_kernel (merge with Kahan sums, thresholding rounds, intersection).
// Stage 2: the UMIs' result lists are deduplicated through a hash table; the DISTINCT lists (thousands, not
// millions) are ranked by feature-string order, and ONE radix sort on (cell ordinal, list rank) puts the UMIs into the
// output order; run lengths are the counts.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "kernels.cuh"
#include "umi_code.hpp"

namespace nb200 {

constexpr int kMaxRounds = 64;   // bound on the reference's `while True` (nimble/utils.py:141)
constexpr int kSmallRows = 8, kSmallNames = 16;   // UMIs up to this size are worked on in thread-local arrays (umi_general_kernel)

// Per-read rows as the kernels see them: padded [n, stride] with a length array (what the alignment kernels write) or
// CSR (what nb200_umi_counts receives).
// Three layouts: padded (off = nullptr: ids + r * stride, nf[r] names), CSR (nf = nullptr: off[r] .. off[r + 1]), and the
// UMI result lists of stage 2 (ids = pool, off = row_off, at = gstart: list of UMI g at pool[row_off[gstart[g]]], nf[g] names;
// at = nullptr for bulk data where UMI g is sorted row g).
struct Rows {
    const int32_t *ids;
    const uint32_t *off;
    const uint32_t *at;
    const uint16_t *nf;
    uint32_t stride;
    __device__ __forceinline__ const int32_t *ptr(uint32_t r) const { return off ? ids + off[at ? at[r] : r] : ids + (uint64_t)r * stride; }
    __device__ __forceinline__ uint32_t len(uint32_t r) const { return nf ? (uint32_t)nf[r] : off[r + 1] - off[r]; }
};

// rows that count (a call, a barcode, a score) -> flag; *max_len <- the longest of them (one atomic per block: the
// alignment kernels used to keep this maximum themselves, 2 M same-address reads per batch)
__global__ void __launch_bounds__(256)
mark_rows_kernel(uint64_t n, const uint64_t *__restrict__ key, Rows rows, const double *__restrict__ score,
                 uint8_t *__restrict__ flag, uint32_t *__restrict__ max_len) {
    __shared__ uint32_t s_max;
    if (threadIdx.x == 0) s_max = 0;
    __syncthreads();
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t len = 0;
    if (i < n) {
        len = rows.len((uint32_t)i);
        bool ok = len > 0;
        if (key && key[i] == NB200_NO_BARCODE) ok = false;
        if (score && score[i] != score[i]) ok = false;
        flag[i] = ok ? 1 : 0;
        if (!ok) len = 0;
    }
    len = __reduce_max_sync(0xFFFFFFFFu, len);
    if ((threadIdx.x & 31) == 0 && len) atomicMax(&s_max, len);
    __syncthreads();
    if (threadIdx.x == 0 && s_max > *(volatile uint32_t *)max_len) atomicMax(max_len, s_max);
}

// CSR input check (nb200_umi_counts): ids in range, ascending inside a row: bit 0 / bit 1 of *err
__global__ void check_rows_kernel(uint64_t n, const uint32_t *__restrict__ off, const uint32_t *__restrict__ ids, uint32_t n_features,
                                  unsigned int *__restrict__ err) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t prev = 0, bad = 0;
    for (uint32_t j = off[i]; j < off[i + 1]; j++) {
        const uint32_t f = ids[j];
        if (f >= n_features) bad |= 1u;
        if (j > off[i] && f < prev) bad |= 2u;
        prev = f;
    }
    if (bad) atomicOr(err, bad);
}

// token-rank columns p0 .. p0+cols-1 of the listed rows packed into one radix key, the earlier position in the more
// significant bits (0 = list shorter than that position): one stable sort on the packed key orders by all of its
// columns at once.  rows: lists addressed by perm[i].
__global__ void gather_tok_kernel(uint32_t m, const uint32_t *__restrict__ perm, Rows rows, uint32_t p0, uint32_t cols, uint32_t bits,
                                  const uint32_t *__restrict__ tok_end, const uint32_t *__restrict__ tok_comma,
                                  uint32_t *__restrict__ out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const uint32_t row = perm[i];
    const uint32_t n = rows.len(row);
    const int32_t *l = rows.ptr(row);
    uint32_t key = 0;
    for (uint32_t j = 0; j < cols; j++) {
        const uint32_t p = p0 + j;
        uint32_t v = 0;
        if (p < n) {
            const uint32_t f = (uint32_t)l[p];
            v = (p == n - 1 ? tok_end[f] : tok_comma[f]) + 1;
        }
        key = (key << bits) | v;
    }
    out[i] = key;
}

// ---- UMI correction (DESIGN.md §2.12): a key-rewrite pre-pass over the selected rows, before the key sort -----------
// Open addressing over 16 B slots, linear probing, load factor <= 0.5.  A slot stores ~key, so that the zeroed table is
// empty: the one key that maps to 0 is NB200_NO_BARCODE, and mark_rows_kernel never selects it.
struct UmiSlot {
    unsigned long long nkey;   // ~key; 0 = empty
    uint32_t count;            // rows with this key
    uint32_t target;           // slot of the key this one is rewritten to (umi_correct_kernel)
};
static_assert(sizeof(UmiSlot) == 16, "one UMI slot is 16 B");

__host__ __device__ __forceinline__ uint32_t umi_slot_hash(uint64_t k) {
    k ^= k >> 33; k *= 0xFF51AFD7ED558CCDull; k ^= k >> 33; k *= 0xC4CEB9FE1A85EC53ull; k ^= k >> 33;
    return (uint32_t)k;
}

// slot of a key present in the table, or 0xFFFFFFFF
__device__ __forceinline__ uint32_t umi_find(const UmiSlot *__restrict__ t, uint32_t mask, uint64_t key) {
    const unsigned long long nk = ~key;
    for (uint32_t s = umi_slot_hash(key) & mask;; s = (s + 1) & mask) {
        const unsigned long long v = t[s].nkey;
        if (v == nk) return s;
        if (v == 0) return 0xFFFFFFFFu;
    }
}

// byte rank of a code digit (A1 C2 G3 T4 N5): the byte order A < C < G < N < T
__host__ __device__ __forceinline__ int umi_digit_rank(uint32_t d) { return d <= 3 ? (int)d - 1 : (d == 4 ? 4 : 3); }

// The UMI's bytes as a fixed-length base-5 number over the byte ranks: for UMIs of one length, numeric order is byte order.
__host__ __device__ __forceinline__ uint32_t umi_byte_value(uint32_t u) {
    uint32_t v = 0, p5 = 1;
    for (uint32_t x = u; x; p5 *= 5) {
        const uint32_t q = (x - 1) / 5;
        v += (uint32_t)umi_digit_rank(x - 5 * q) * p5;
        x = q;
    }
    return v;
}

// Every one-substitution neighbour of code u (1 <= u <= kUmiCodeMax): each position, each of A C G T other than the base
// there (N positions included), never N.  f(code, byte value) with byte value as umi_byte_value would give it.  A neighbour
// is one add to the code, (d' - d) * 5^p, and one to the byte value.  (Host callers pass host lambdas: nb200_umi_neighbours.)
#pragma nv_exec_check_disable
template <class F>
__host__ __device__ __forceinline__ void umi_for_each_neighbour(uint32_t u, uint32_t bv, F &&f) {
    uint32_t p5 = 1;
    for (uint32_t x = u; x; p5 *= 5) {
        const uint32_t q = (x - 1) / 5, d = x - 5 * q;
        const int rd = umi_digit_rank(d);
        for (uint32_t e = 1; e <= 4; e++) {
            if (e == d) continue;
            f((uint32_t)((int64_t)u + ((int64_t)e - (int64_t)d) * p5), (uint32_t)((int64_t)bv + (int64_t)(umi_digit_rank(e) - rd) * p5));
        }
        x = q;
    }
}

// one thread per selected row: its key into the table, one more row for it
__global__ void __launch_bounds__(256)
umi_count_kernel(uint32_t m, const uint64_t *__restrict__ key, UmiSlot *__restrict__ t, uint32_t mask) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const uint64_t k = key[i];
    const unsigned long long nk = ~k;
    for (uint32_t s = umi_slot_hash(k) & mask;; s = (s + 1) & mask) {
        unsigned long long v = *(volatile unsigned long long *)&t[s].nkey;
        if (v == 0) v = atomicCAS(&t[s].nkey, 0ull, nk);
        if (v == 0 || v == nk) { atomicAdd(&t[s].count, 1u); return; }
    }
}

// one thread per slot: target = the maximum of (rows, bytes) over the key itself and its present one-substitution
// neighbours in the same cell, from the counts as umi_count_kernel left them (no slot's count changes here, so targets do
// not depend on thread order).  Keys whose UMI is not a code (interned) keep themselves.  *corrected += keys whose target
// is another key (one atomic per block).
__global__ void __launch_bounds__(256)
umi_correct_kernel(uint32_t tsize, UmiSlot *__restrict__ t, uint32_t mask, uint32_t *__restrict__ corrected) {
    const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    int moved = 0;
    if (s < tsize) {
        const unsigned long long nk = t[s].nkey;
        uint32_t best = s;
        if (nk) {
            const uint64_t k = ~nk;
            const uint32_t u = (uint32_t)k;
            if (u >= 1 && u <= kUmiCodeMax) {
                const uint64_t cell = k & 0xFFFFFFFF00000000ull;
                uint32_t best_n = t[s].count, best_bv = umi_byte_value(u);
                umi_for_each_neighbour(u, best_bv, [&](uint32_t v, uint32_t bv) {
                    const uint32_t o = umi_find(t, mask, cell | v);
                    if (o == 0xFFFFFFFFu) return;
                    const uint32_t n = t[o].count;
                    if (n > best_n || (n == best_n && bv > best_bv)) { best = o; best_n = n; best_bv = bv; }
                });
            }
            t[s].target = best;
            moved = best != s;
        }
    }
    moved = __syncthreads_count(moved);
    if (threadIdx.x == 0 && moved) atomicAdd(corrected, (uint32_t)moved);
}

// one thread per selected row (key[i] is row perm[i]'s key): out[perm[i]] = the key of its slot's target.  out is
// indexed like the caller's key array, so every later reader of a row's key (gather_key64_kernel, also on the second key
// sort of the large-group path) sees the rewritten key.
__global__ void __launch_bounds__(256)
umi_rewrite_kernel(uint32_t m, const uint32_t *__restrict__ perm, const uint64_t *__restrict__ key, const UmiSlot *__restrict__ t,
                   uint32_t mask, uint64_t *__restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const uint32_t s = umi_find(t, mask, key[i]);
    out[perm[i]] = ~t[t[s].target].nkey;
}

__global__ void gather_key64_kernel(uint32_t m, const uint32_t *__restrict__ perm, const uint64_t *__restrict__ key,
                                    uint64_t *__restrict__ out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    out[i] = key[perm[i]];
}

// sorted keys -> head flags, and names per sorted row (input of the exclusive scan that lays out the per-UMI pools)
__global__ void key_heads_kernel(uint32_t m, const uint64_t *__restrict__ sorted_key, const uint32_t *__restrict__ perm, Rows rows,
                                 uint8_t *__restrict__ head, uint32_t *__restrict__ row_n) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > m) return;
    if (i == m) { row_n[i] = 0; return; }                    // scan sentinel: row_off[m] = total names
    head[i] = (i == 0 || sorted_key[i] != sorted_key[i - 1]) ? 1 : 0;
    row_n[i] = rows.len(perm[i]);
}

__device__ __forceinline__ bool same_list(const int32_t *a, uint32_t na, const int32_t *b, uint32_t nb) {
    if (na != nb) return false;
    for (uint32_t j = 0; j < na; j++) if (a[j] != b[j]) return false;
    return true;
}

// order of two rows by the byte order of their comma-joined feature strings: token ranks position by position,
// name+NUL for the last name of a row, name+',' otherwise
__device__ __forceinline__ int compare_rows(const int32_t *la, uint32_t na, const int32_t *lb, uint32_t nb,
                                            const uint32_t *__restrict__ tok_end, const uint32_t *__restrict__ tok_comma) {
    const uint32_t mn = na < nb ? na : nb;
    for (uint32_t p = 0; p < mn; p++) {
        const uint32_t ta = (p == na - 1) ? tok_end[la[p]] : tok_comma[la[p]];
        const uint32_t tb = (p == nb - 1) ? tok_end[lb[p]] : tok_comma[lb[p]];
        if (ta != tb) return ta < tb ? -1 : 1;
    }
    return na < nb ? -1 : (na > nb ? 1 : 0);       // only reached for empty rows
}

// dev[0] = number of (cell, umi) groups (DeviceSelect wrote it); dev[1] <- largest group (decides between the per-group
// sort and the global token sort).  Launched over m threads, the group count is only known on the device.
__global__ void max_group_kernel(const uint32_t *__restrict__ dev, const uint32_t *__restrict__ gstart, uint32_t m, unsigned int *__restrict__ out) {
    const uint32_t n_groups = dev[0];
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t sz = 0;
    if (g < n_groups) sz = ((g + 1 < n_groups) ? gstart[g + 1] : m) - gstart[g];
    sz = __reduce_max_sync(0xFFFFFFFFu, sz);
    if ((threadIdx.x & 31) == 0 && sz > *(volatile unsigned int *)out) atomicMax(out, sz);
}

// rows of one (cell, umi) group -> ascending feature-string order, stable (insertion sort on the permutation;
// groups are a handful of rows, the caller falls back to the global sort when one exceeds kLocalSortMax)
constexpr uint32_t kLocalSortMax = 48;
__global__ void __launch_bounds__(128)
group_sort_kernel(uint32_t n_groups, const uint32_t *__restrict__ gstart, uint32_t m, uint32_t *__restrict__ perm, Rows rows,
                  const uint32_t *__restrict__ tok_end, const uint32_t *__restrict__ tok_comma) {
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_groups) return;
    const uint32_t g0 = gstart[g], g1 = (g + 1 < n_groups) ? gstart[g + 1] : m;
    for (uint32_t i = g0 + 1; i < g1; i++) {
        const uint32_t r = perm[i];
        const int32_t *lr = rows.ptr(r);
        const uint32_t nr = rows.len(r);
        uint32_t j = i;
        while (j > g0) {
            const uint32_t q = perm[j - 1];
            if (compare_rows(rows.ptr(q), rows.len(q), lr, nr, tok_end, tok_comma) <= 0) break;   // stable
            perm[j] = q;
            j--;
        }
        perm[j] = r;
    }
}

__device__ inline void heap_sort_u32(uint32_t *a, int n) {
    for (int start = n / 2 - 1; start >= 0; start--) {
        int root = start;
        for (;;) {
            int child = 2 * root + 1;
            if (child >= n) break;
            if (child + 1 < n && a[child] < a[child + 1]) child++;
            if (a[root] >= a[child]) break;
            uint32_t t = a[root]; a[root] = a[child]; a[child] = t;
            root = child;
        }
    }
    for (int end = n - 1; end > 0; end--) {
        uint32_t t = a[0]; a[0] = a[end]; a[end] = t;
        int root = 0;
        for (;;) {
            int child = 2 * root + 1;
            if (child >= end) break;
            if (child + 1 < end && a[child] < a[child + 1]) child++;
            if (a[root] >= a[child]) break;
            uint32_t u = a[root]; a[root] = a[child]; a[child] = u;
            root = child;
        }
    }
}

__device__ __forceinline__ int find_u32(const uint32_t *U, int nu, uint32_t v) {
    int lo = 0, hi = nu - 1;
    while (lo < hi) {
        int mid = (lo + hi) >> 1;
        if (U[mid] < v) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// Per-UMI state.  Pools are laid out by row_off (exclusive scan of the names per sorted row): the UMI whose rows are
// sorted positions [g0, g1) owns pool entries [row_off[g0], row_off[g1]) — room for its feature universe and for its
// result list, without any atomic and without padding to the longest row.
struct UmiScratch {
    const uint32_t *row_off;  // [m + 1]
    uint32_t *rep;            // [m]  merged row -> representative sorted position
    double *S;                // [m]  merged score
    uint32_t *U;              // [T]  feature universe of the group
    double *fs, *fc;          // [T]  Kahan sum / compensation per feature
    uint8_t *flags;           // [T]  bit0 present, bit1 drop-now, bit2 keep
};

struct UmiOut {
    uint32_t *cell;           // [G]
    uint16_t *n;              // [G]  names of the result list (0: the UMI counts nowhere)
    int32_t *list;            // [T]  result list of group g at row_off[gstart[g]]
};

// nimble/utils.py:125-131 and :158-165 — feature scores from the ORIGINAL merged rows minus the
// names flagged drop-now.  Kahan per feature in order of appearance == pandas group_sum.
__device__ inline bool umi_scores(int m, const uint32_t *rep, const double *S, const uint32_t *perm, const Rows &rows,
                                  const uint32_t *U, int nu, double *fs, double *fc, uint8_t *flags, double &total_out) {
    double total = 0.0;
    bool any = false;
    for (int j = 0; j < nu; j++) { fs[j] = 0.0; fc[j] = 0.0; flags[j] &= ~1; }
    for (int d = 0; d < m; d++) {
        const uint32_t row = perm[rep[d]];
        const int32_t *l = rows.ptr(row);
        const int n = (int)rows.len(row);
        int len = 0;
        for (int j = 0; j < n; j++) if (!(flags[find_u32(U, nu, (uint32_t)l[j])] & 2)) len++;
        if (!len) continue;
        any = true;
        const double share = S[d] / (double)len;
        total += S[d];
        for (int j = 0; j < n; j++) {
            const int q = find_u32(U, nu, (uint32_t)l[j]);
            if (flags[q] & 2) continue;
            const double y = share - fc[q];
            const double t = fs[q] + y;
            double c = (t - fs[q]) - y;
            if (c != c) c = 0.0;
            fc[q] = c; fs[q] = t;
            flags[q] |= 1;
        }
    }
    total_out = total;
    return any;
}

// One thread per (cell, umi) group; rows arrive sorted by (key, feature-string order, input order).  Settles the UMIs
// whose rows all carry the same list without duplicate names: every feature then has the same ratio (S/len)/S, computed
// exactly as the general path would (Kahan in input order, pandas groupby-sum, __main__.py:251).  The others are
// appended to `slow` (dev[2] counts them) for umi_general_kernel.
__global__ void __launch_bounds__(128)
umi_simple_kernel(uint32_t n_groups, const uint32_t *__restrict__ gstart, uint32_t m, const uint32_t *__restrict__ perm,
                  const uint64_t *__restrict__ sorted_key, Rows rows, const double *__restrict__ score, double threshold, int disable,
                  const uint32_t *__restrict__ row_off, UmiOut out, uint32_t *__restrict__ slow, uint32_t *__restrict__ dev) {
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    bool general = false;
    if (g < n_groups) {
        const uint32_t g0 = gstart[g], g1 = (g + 1 < n_groups) ? gstart[g + 1] : m;
        const uint32_t ra = perm[g0];
        const int32_t *l = rows.ptr(ra);
        const uint32_t n = rows.len(ra);
        double s = 0.0, c = 0.0;
        bool one = true;
        for (uint32_t u = g0; u < g1 && one; u++) {
            const uint32_t rb = perm[u];
            if (u > g0 && !same_list(l, n, rows.ptr(rb), rows.len(rb))) { one = false; break; }
            const double v = score ? score[rb] : 1.0;
            const double y = v - c, tt = s + y;
            c = (tt - s) - y;
            if (c != c) c = 0.0;
            s = tt;
        }
        bool dup = false;
        for (uint32_t j = 1; j < n; j++) dup |= (l[j] == l[j - 1]);
        general = !one || dup;
        if (!general) {
            bool keep_all = true;
            if (!disable) {
                const double share = s / (double)n;
                const double ratio = share / s;
                keep_all = !(ratio < threshold);
            }
            int32_t *dst = out.list + row_off[g0];
            if (keep_all) for (uint32_t j = 0; j < n; j++) dst[j] = l[j];
            out.cell[g] = (uint32_t)(sorted_key[g0] >> 32);
            out.n[g] = (uint16_t)(keep_all ? n : 0);
        }
    }
    const unsigned gb = __ballot_sync(0xFFFFFFFFu, general);
    if (gb) {
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(&dev[2], (uint32_t)__popc(gb));
        base = __shfl_sync(0xFFFFFFFFu, base, 0);
        if (general) slow[base + __popc(gb & ((1u << lane) - 1))] = g;
    }
}

// The general path (nimble/utils.py:119-224), one thread per listed UMI: the list is compact, so the threads of a warp
// all walk a multi-row UMI.
__global__ void __launch_bounds__(128)
umi_general_kernel(const uint32_t *__restrict__ slow, const uint32_t *__restrict__ dev, uint32_t n_groups, const uint32_t *__restrict__ gstart,
                   uint32_t m, const uint32_t *__restrict__ perm, const uint64_t *__restrict__ sorted_key, Rows rows,
                   const double *__restrict__ score, double threshold, int disable, UmiScratch sc, UmiOut out,
                   Counters *__restrict__ ctr) {
    const uint32_t n_slow = dev[2];
    for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < n_slow; t += gridDim.x * blockDim.x) {
        const uint32_t g = slow[t];
        const uint32_t g0 = gstart[g], g1 = (g + 1 < n_groups) ? gstart[g + 1] : m;
        const uint32_t p0 = sc.row_off[g0];
        // working set of the UMI: thread-local arrays when it is small (nearly always: a few rows, a dozen names; local
        // memory is interleaved per thread and L1-resident), its slice of the global pools otherwise
        uint32_t l_rep[kSmallRows], l_U[kSmallNames];
        double l_S[kSmallRows], l_fs[kSmallNames], l_fc[kSmallNames];
        uint8_t l_flags[kSmallNames];
        const bool small = g1 - g0 <= (uint32_t)kSmallRows && sc.row_off[g1] - p0 <= (uint32_t)kSmallNames;
        uint32_t *rep = small ? l_rep : sc.rep + g0;
        double *S = small ? l_S : sc.S + g0;
        uint32_t *U = small ? l_U : sc.U + p0;
        double *fs = small ? l_fs : sc.fs + p0, *fc = small ? l_fc : sc.fc + p0;
        uint8_t *flags = small ? l_flags : sc.flags + p0;
        // merged rows: runs of identical lists; Kahan in input order (pandas groupby-sum, __main__.py:251)
        int md = 0;
        for (uint32_t a = g0; a < g1;) {
            const uint32_t ra = perm[a];
            double s = 0.0, c = 0.0;
            uint32_t u = a;
            while (u < g1) {
                const uint32_t rb = perm[u];
                if (!same_list(rows.ptr(ra), rows.len(ra), rows.ptr(rb), rows.len(rb))) break;
                const double v = score ? score[rb] : 1.0;
                const double y = v - c, tt = s + y;
                c = (tt - s) - y;
                if (c != c) c = 0.0;
                s = tt;
                u++;
            }
            rep[md] = a; S[md] = s; md++;
            a = u;
        }
        // feature universe
        int nu = 0;
        for (int d = 0; d < md; d++) {
            const uint32_t row = perm[rep[d]];
            const int32_t *l = rows.ptr(row);
            const int n = (int)rows.len(row);
            for (int j = 0; j < n; j++) U[nu++] = (uint32_t)l[j];
        }
        heap_sort_u32(U, nu);
        {
            int w = 0;
            for (int j = 0; j < nu; j++) if (j == 0 || U[j] != U[j - 1]) U[w++] = U[j];
            nu = w;
        }
        for (int j = 0; j < nu; j++) flags[j] = 0;
        if (disable) {
            for (int j = 0; j < nu; j++) flags[j] = 4;
        } else {
            double total = 0.0;
            bool any = umi_scores(md, rep, S, perm, rows, U, nu, fs, fc, flags, total);
            bool done = false;
            for (int round = 0; round < kMaxRounds && !done; round++) {
                if (!any) { done = true; break; }          // keep = {}
                int nd = 0;
                for (int j = 0; j < nu; j++) {
                    flags[j] &= ~2;
                    if (!(flags[j] & 1)) continue;
                    const double ratio = fs[j] / total;       // IEEE: x/0 = inf, 0/0 = nan -> never < thr
                    if (ratio < threshold) { flags[j] |= 2; nd++; }
                }
                if (nd == 0) {
                    for (int j = 0; j < nu; j++) if (flags[j] & 1) flags[j] |= 4;
                    done = true;
                    break;
                }
                any = umi_scores(md, rep, S, perm, rows, U, nu, fs, fc, flags, total);
            }
            if (!done && any) for (int j = 0; j < nu; j++) if (flags[j] & 1) flags[j] |= 4;
        }
        // per merged row: filtered = sorted(set(row) & keep); empty rows vanish; intersect the rest
        int32_t *inter = out.list + p0;
        int ni = -1;
        for (int d = 0; d < md; d++) {
            const uint32_t row = perm[rep[d]];
            const int32_t *l = rows.ptr(row);
            const int n = (int)rows.len(row);
            if (ni < 0) {
                int w = 0;
                for (int j = 0; j < n; j++) {
                    if (!(flags[find_u32(U, nu, (uint32_t)l[j])] & 4)) continue;
                    if (w && inter[w - 1] == l[j]) continue;
                    inter[w++] = l[j];
                }
                if (w) ni = w;
            } else {
                // does the row keep anything at all?  (rows left empty are dropped, utils.py:205)
                bool nonempty = false;
                for (int j = 0; j < n && !nonempty; j++) nonempty = (flags[find_u32(U, nu, (uint32_t)l[j])] & 4) != 0;
                if (!nonempty) continue;
                int w = 0;
                for (int x = 0; x < ni; x++) {
                    bool in = false;
                    for (int j = 0; j < n && !in; j++) in = (l[j] == inter[x]);   // kept by construction
                    if (in) inter[w++] = inter[x];
                }
                ni = w;
            }
        }
        if (ni == 0) atomicAdd(&ctr->dropped_empty, 1ull);
        out.cell[g] = (uint32_t)(sorted_key[g0] >> 32);
        out.n[g] = (uint16_t)(ni > 0 ? ni : 0);
    }
}

// bulk data (no barcodes): every called read is its own "UMI" with cell 0; its list is the row itself
__global__ void bulk_rows_kernel(uint32_t m, const uint32_t *__restrict__ perm, Rows rows, const uint32_t *__restrict__ row_off, UmiOut out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const uint32_t row = perm[i];
    const uint32_t n = rows.len(row);
    const int32_t *l = rows.ptr(row);
    int32_t *dst = out.list + row_off[i];
    out.cell[i] = 0;
    out.n[i] = (uint16_t)n;
    for (uint32_t j = 0; j < n; j++) dst[j] = l[j];
}

// ---- stage 2 ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t hash_list(const int32_t *l, uint32_t n) {
    uint32_t h = 0x9E3779B9u ^ n;
    for (uint32_t j = 0; j < n; j++) { h ^= (uint32_t)l[j]; h *= 0x85EBCA6Bu; h ^= h >> 15; }
    h *= 0xC2B2AE35u;
    return h ^ (h >> 16);
}

// Every UMI with a result finds the representative of its list: open addressing over `table` (0 = empty, g + 1 = the UMI
// that claimed the slot), lists compared in full.  rep_of[g] = g for the representatives, 0xFFFFFFFF for UMIs without
// a result.  Which UMI of a list becomes the representative depends on timing; nothing downstream depends on which.
__global__ void dedupe_lists_kernel(uint32_t G, Rows lists, uint32_t *__restrict__ table, uint32_t mask, uint32_t *__restrict__ rep_of,
                                    uint8_t *__restrict__ is_rep) {
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= G) return;
    const uint32_t n = lists.len(g);
    if (!n) { rep_of[g] = 0xFFFFFFFFu; is_rep[g] = 0; return; }
    const int32_t *l = lists.ptr(g);
    uint32_t s = hash_list(l, n) & mask;
    for (;;) {
        uint32_t cur = *(volatile uint32_t *)(table + s);
        if (cur == 0) {
            cur = atomicCAS(table + s, 0u, g + 1);
            if (cur == 0) { rep_of[g] = g; is_rep[g] = 1; return; }
        }
        const uint32_t o = cur - 1;
        // the claimant's list was complete before this kernel started (the umi kernels ran earlier on the stream)
        if (same_list(l, n, lists.ptr(o), lists.len(o))) { rep_of[g] = o; is_rep[g] = 0; return; }
        s = (s + 1) & mask;
    }
}

// names per sorted row for bulk data (the tagged path gets them from key_heads_kernel)
__global__ void row_len_kernel(uint32_t m, const uint32_t *__restrict__ perm, Rows rows, uint32_t *__restrict__ row_n) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > m) return;
    row_n[i] = i < m ? rows.len(perm[i]) : 0u;
}

// UMIs arrive in (cell, umi) order: flag where the cell changes (scan -> cell ordinal), count the UMIs with a result
__global__ void cell_heads_kernel(uint32_t G, const uint32_t *__restrict__ cell, uint32_t *__restrict__ head) {
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= G) return;
    head[g] = (g > 0 && cell[g] != cell[g - 1]) ? 1u : 0u;
}

__global__ void scatter_rank_kernel(uint32_t D, const uint32_t *__restrict__ sorted_rep, uint32_t *__restrict__ rank_of) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < D) rank_of[sorted_rep[i]] = i;
}

// sort key of a UMI: (cell ordinal << rank_bits) | rank of its list; UMIs without a result get the sentinel above all keys
__global__ void umi_keys_kernel(uint32_t G, const uint32_t *__restrict__ cell_ord, const uint32_t *__restrict__ rep_of,
                                const uint32_t *__restrict__ rank_of, uint32_t rank_bits, uint64_t sentinel,
                                uint64_t *__restrict__ key, uint32_t *__restrict__ val) {
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= G) return;
    const uint32_t r = rep_of[g];
    key[g] = r == 0xFFFFFFFFu ? sentinel : (((uint64_t)cell_ord[g] << rank_bits) | rank_of[r]);
    val[g] = g;
}

// run heads over the sorted keys; dev[4] += names of the run heads' lists (size of the id array)
__global__ void __launch_bounds__(256)
run_heads_kernel(uint32_t G, const uint64_t *__restrict__ key, const uint32_t *__restrict__ val, uint64_t sentinel,
                 const uint16_t *__restrict__ n, uint8_t *__restrict__ head, uint32_t *__restrict__ dev) {
    __shared__ uint32_t s_ids, s_live;
    if (threadIdx.x == 0) { s_ids = 0; s_live = 0; }
    __syncthreads();
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    bool h = false, live = false;
    uint32_t ids = 0;
    if (i < G) {
        const uint64_t k = key[i];
        live = k != sentinel;
        h = live && (i == 0 || k != key[i - 1]);
        head[i] = h ? 1 : 0;
        if (h) ids = n[val[i]];
    }
    ids = __reduce_add_sync(0xFFFFFFFFu, ids);
    const unsigned lb = __ballot_sync(0xFFFFFFFFu, live);
    if ((threadIdx.x & 31) == 0) {                                   // one global atomic per block, not per warp
        if (ids) atomicAdd(&s_ids, ids);
        if (lb) atomicAdd(&s_live, (uint32_t)__popc(lb));
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (s_ids) atomicAdd(&dev[4], s_ids);
        if (s_live) atomicAdd(&dev[5], s_live);                      // UMIs with a result = end of the last run
    }
}

// run i -> (cell, count, n_feat) ; n_feat feeds the exclusive scan that lays out the CSR ids
__global__ void emit_counts_kernel(uint32_t n_out, const uint32_t *__restrict__ starts, const uint32_t *__restrict__ dev,
                                   const uint32_t *__restrict__ val, const uint32_t *__restrict__ cell, const uint16_t *__restrict__ n,
                                   uint32_t *__restrict__ o_cell, uint32_t *__restrict__ o_count, uint32_t *__restrict__ o_n) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n_out) return;
    if (i == n_out) { o_n[i] = 0; return; }          // scan sentinel -> o_off[n_out] = total ids
    const uint32_t s = starts[i], e = (i + 1 < n_out) ? starts[i + 1] : dev[5];
    const uint32_t g = val[s];
    o_cell[i] = cell[g];
    o_count[i] = e - s;
    o_n[i] = n[g];
}

__global__ void emit_ids_kernel(uint32_t n_out, const uint32_t *__restrict__ starts, const uint32_t *__restrict__ val, Rows lists,
                                const uint32_t *__restrict__ o_off, uint32_t *__restrict__ o_ids) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_out) return;
    const int32_t *l = lists.ptr(val[starts[i]]);
    const uint32_t a = o_off[i], b = o_off[i + 1];
    for (uint32_t j = a; j < b; j++) o_ids[j] = (uint32_t)l[j - a];
}

// ---- counts from files (nb200_align_files_counts): the row store ---------------------------------------------------
// A slab's rows that reach the UMI stage are appended to the library's row store behind its calling kernels; the rows
// are the ones `report` keeps of the per-read TSV: a call, a cell and a UMI (no NB200_NO_BARCODE), and not a single
// feature whose name pandas reads as NaN (na_name[f], pandas_na.hpp).

// read i -> (1 << 32 | names) when its row counts, else 0; entry n = 0 (the exclusive scan's total); *called += reads with
// a call
__global__ void __launch_bounds__(256)
row_flag_kernel(uint32_t n, const uint64_t *__restrict__ key, const nb200_read_result *__restrict__ res, const int32_t *__restrict__ feats,
                uint32_t mh, const uint8_t *__restrict__ na_name, uint64_t *__restrict__ val, unsigned long long *__restrict__ called) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    int c = 0;
    if (i < n) {
        const uint32_t k = res[i].n_feat;
        c = k > 0;
        bool keep = k > 0 && key[i] != NB200_NO_BARCODE;
        if (keep && k == 1 && na_name[feats[(uint64_t)i * mh]]) keep = false;
        val[i] = keep ? ((1ull << 32) | k) : 0ull;
    } else if (i == n) {
        val[i] = 0ull;
    }
    c = __syncthreads_count(c);
    if (threadIdx.x == 0 && c) atomicAdd(called, (unsigned long long)c);
}

// pos = exclusive scan of row_flag_kernel's values: (row, id) offsets of read i inside the slab's segment; the segment
// starts where the store ends (hdr[0] rows, hdr[1] ids: device-side, so that no host round trip sits between slabs)
__global__ void __launch_bounds__(256)
row_scatter_kernel(uint32_t n, const uint64_t *__restrict__ key, const int32_t *__restrict__ feats, uint32_t mh,
                   const uint64_t *__restrict__ pos, const unsigned long long *__restrict__ hdr,
                   uint64_t *__restrict__ s_key, uint32_t *__restrict__ s_nf, int32_t *__restrict__ s_ids) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t a = pos[i], b = pos[i + 1];
    if ((a >> 32) == (b >> 32)) return;
    const uint64_t r = hdr[0] + (a >> 32), p = hdr[1] + (a & 0xFFFFFFFFull);
    const uint32_t k = (uint32_t)(b - a);                  // (1 << 32 | k) apart
    s_key[r] = key[i];
    s_nf[r] = k;
    const int32_t *f = feats + (uint64_t)i * mh;
    for (uint32_t j = 0; j < k; j++) s_ids[p + j] = f[j];
}

// segment record seg = {first row, rows, first id, ids, (called)}; the store's end moves past it
__global__ void row_advance_kernel(const uint64_t *__restrict__ total, unsigned long long *__restrict__ hdr, unsigned long long *__restrict__ seg) {
    const uint64_t t = *total, rows = t >> 32, ids = t & 0xFFFFFFFFull;
    seg[0] = hdr[0]; seg[1] = rows; seg[2] = hdr[1]; seg[3] = ids;
    hdr[0] += rows; hdr[1] += ids;
}

// cell id (first-seen order of the host dictionary) -> rank of its CB string: the UMI stage orders cells by key, and
// the counts TSV orders them by CB bytes
__global__ void __launch_bounds__(256)
cell_rank_kernel(uint64_t n, uint64_t *__restrict__ key, const uint32_t *__restrict__ rank) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint64_t k = key[i];
    key[i] = ((uint64_t)rank[k >> 32] << 32) | (k & 0xFFFFFFFFull);
}

}  // namespace nb200
