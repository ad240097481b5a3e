// Checksum of the sections of an index file (library.cpp), shared with the device check of a loaded image
// (engine.cu): the sum mod 2^64 over 64-bit words w_i of splitmix64(w_i ^ i * C).  The sum does not depend on the order
// of its terms, so host threads and a grid-stride kernel can split it freely; splitmix64 is a bijection and i * C
// differs per word, so changing any single word always changes the sum.
#pragma once
#include <cstdint>

#ifdef __CUDACC__
#define NB200_SUM_HD __host__ __device__ __forceinline__
#else
#define NB200_SUM_HD inline
#endif

namespace nb200 {

NB200_SUM_HD uint64_t image_word_sum(uint64_t w, uint64_t i) {
    uint64_t z = w ^ (i * 0x9E3779B97F4A7C15ull);
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

}  // namespace nb200
