// Bucket addressing of the k-mer table, shared by the host builder (library.cpp) and the kernels (kernels.cuh).
// 32-bit arithmetic only: the probe kernel is instruction-issue bound, a 64-bit multiply costs four instructions.
#pragma once
#include <cstdint>

#ifdef __CUDACC__
#define NB200_HD __host__ __device__ __forceinline__
#else
#define NB200_HD inline
#endif

namespace nb200 {

// canonical k-mer (lo, hi halves) -> mixed 32-bit value; the first bucket uses its upper bits (multiply-high by
// the bucket count), the second bucket a second mix of it and the key.  Index files store tables built with these:
// any change to kmer_mix or the bucket functions must bump kIndexVersion (library.hpp).
NB200_HD uint32_t kmer_mix(uint32_t clo, uint32_t chi) {
    uint32_t a = clo * 0x9E3779B1u + chi * 0x85EBCA77u;
    a ^= a >> 15;
    a *= 0xC2B2AE3Du;
    a ^= a >> 13;
    return a;
}
NB200_HD uint32_t mulhi32(uint32_t a, uint32_t b) {
#ifdef __CUDA_ARCH__
    return __umulhi(a, b);
#else
    return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}
NB200_HD uint32_t kmer_bucket1(uint32_t mix, uint32_t n_buckets) { return mulhi32(mix, n_buckets); }
NB200_HD uint32_t kmer_bucket2(uint32_t mix, uint32_t clo, uint32_t b1, uint32_t n_buckets) {
    uint32_t h = (mix ^ clo) * 0x27D4EB2Fu;
    h ^= h >> 15;
    h *= 0x165667B1u;
    const uint32_t b2 = mulhi32(h, n_buckets);
    return b2 != b1 ? b2 : (b1 + 1 == n_buckets ? 0u : b1 + 1);
}

}  // namespace nb200
