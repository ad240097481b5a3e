// The one UMI code of the UMI stage.  `report` only compares UMIs for equality, so a UMI needs no dictionary when it is
// short: an ACGTN string of 1..13 bases is its bijective base-5 value (A C G T N = digits 1..5, the last base least
// significant), below 2^31 and injective across lengths.  Every other UMI is interned by its reader with bit 31 set.
// The device decodes this code to correct UMIs (agg.cuh: umi_correct_kernel, DESIGN.md §2.12), so stream.cpp (files),
// report.cpp (per-read TSV) and the Python mirror (frontend.umi_code) must all encode this way.
#pragma once
#include <array>
#include <cstdint>
#include <string_view>

namespace nb200 {

constexpr int kUmiCodeBases = 13;
constexpr uint32_t kUmiCodeMax = 1525878905u;      // NNNNNNNNNNNNN: 5 * (5^13 - 1) / 4
constexpr uint32_t kUmiInterned = 0x80000000u;     // bit of an interned UMI id

// bijective base 5 of an ACGTN string of 1..13 bases; false for anything else
static inline bool umi_code(std::string_view s, uint32_t &x) {
    static const auto digit = [] { std::array<uint8_t, 256> d{}; d['A'] = 1; d['C'] = 2; d['G'] = 3; d['T'] = 4; d['N'] = 5; return d; }();
    if (s.empty() || s.size() > (size_t)kUmiCodeBases) return false;
    x = 0;
    for (char ch : s) {
        const uint32_t d = digit[(unsigned char)ch];
        if (!d) return false;
        x = x * 5u + d;
    }
    return true;
}

}  // namespace nb200
