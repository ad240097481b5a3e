// Device side of `report -s` (summarize_fields, nimble/__main__.py:291-297; host side csrc/summarize.cpp, DESIGN.md §2.13).
// Input per column: the rows (ascending) whose UMI and cell are present and the cell's value key (equal typed values,
// equal keys: exact, no hash).  Stable radix sorts by value key, then by UMI rank, put each (UMI, value) pair's rows
// together in file order; a run of them gives the pair's count and first row.  The runs are then ordered inside their
// UMI by count descending, first row ascending (Python's stable sort on -count over first appearances) by two more
// stable sorts.  The orchestration (nb200_summarize_file, engine.cu) keeps the sorts in CUB.
#pragma once
#include <cstdint>

namespace nb200 {

// UMI keys sorted: head[i] = 1 where a new UMI starts (its inclusive sum, minus one, is the UMI's rank in typed order)
__global__ void sum_umi_head_kernel(uint32_t m, const uint64_t *__restrict__ key, uint32_t *__restrict__ head) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < m) head[i] = i == 0 || key[i] != key[i - 1];
}

// rank of every row's UMI, and each UMI's first row (the stable sort keeps rows ascending inside a UMI)
__global__ void sum_umi_rank_kernel(uint32_t m, const uint32_t *__restrict__ scan, const uint32_t *__restrict__ row,
                                    uint32_t *__restrict__ rank_of_row, uint32_t *__restrict__ umi_first) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const uint32_t r = scan[i] - 1;
    rank_of_row[row[i]] = r;
    if (i == 0 || scan[i - 1] != scan[i]) umi_first[r] = row[i];
}

// value-sorted rows -> their UMI ranks (key of the second sort) and positions (its payload)
__global__ void sum_gather_rank_kernel(uint32_t m, const uint32_t *__restrict__ row, const uint32_t *__restrict__ rank_of_row,
                                       uint32_t *__restrict__ urank, uint32_t *__restrict__ pos) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    urank[i] = rank_of_row[row[i]];
    pos[i] = i;
}

// (UMI rank, value key) order: flag[i] = 1 where a (UMI, value) run starts; the rows in that order
__global__ void sum_run_head_kernel(uint32_t m, const uint32_t *__restrict__ urank, const uint32_t *__restrict__ pos,
                                    const uint64_t *__restrict__ vkey, const uint32_t *__restrict__ vrow,
                                    uint8_t *__restrict__ flag, uint32_t *__restrict__ row_out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const uint32_t j = pos[i];
    row_out[i] = vrow[j];
    flag[i] = i == 0 || urank[i] != urank[i - 1] || vkey[j] != vkey[pos[i - 1]];
}

// per run q: its UMI rank, count and first row, the order key (cmask - count) << rbits | first row (count descending,
// then first appearance), and its index as payload
__global__ void sum_run_kernel(uint32_t r, uint32_t m, const uint32_t *__restrict__ head, const uint32_t *__restrict__ urank,
                               const uint32_t *__restrict__ row, uint32_t cmask, int rbits, uint32_t *__restrict__ run_u,
                               uint32_t *__restrict__ run_count, uint32_t *__restrict__ run_first, uint64_t *__restrict__ okey,
                               uint32_t *__restrict__ idx) {
    const uint32_t q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= r) return;
    const uint32_t s = head[q], e = q + 1 < r ? head[q + 1] : m, cnt = e - s;
    run_u[q] = urank[s];
    run_count[q] = cnt;
    run_first[q] = row[s];
    okey[q] = ((uint64_t)(cmask - cnt) << rbits) | row[s];
    idx[q] = q;
}

// runs in order-key order -> their UMI ranks (key of the last sort) and positions
__global__ void sum_gather_run_umi_kernel(uint32_t r, const uint32_t *__restrict__ idx, const uint32_t *__restrict__ run_u,
                                          uint32_t *__restrict__ u_out, uint32_t *__restrict__ pos) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= r) return;
    u_out[p] = run_u[idx[p]];
    pos[p] = p;
}

// the runs in output order: out = [UMI rank x r | count x r | first row x r]
__global__ void sum_out_kernel(uint32_t r, const uint32_t *__restrict__ u_sorted, const uint32_t *__restrict__ pos,
                               const uint32_t *__restrict__ idx, const uint32_t *__restrict__ run_count,
                               const uint32_t *__restrict__ run_first, uint32_t *__restrict__ out) {
    const uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= r) return;
    const uint32_t q = idx[pos[p]];
    out[p] = u_sorted[p];
    out[(size_t)r + p] = run_count[q];
    out[2 * (size_t)r + p] = run_first[q];
}

}  // namespace nb200
