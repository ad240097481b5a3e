// Host file code outside the streaming pipeline: whole-file reads, the 10x one-pass route's per-read TSV, fastq-to-bam, report.
#pragma once
#include <chrono>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/nimble_b200.h"

namespace nb200 {

struct IoError : std::runtime_error { using std::runtime_error::runtime_error; };

struct PhaseTimer {                       // NB200_TRACE=1: phase times of the host file code on stderr
    bool on = getenv("NB200_TRACE") != nullptr;
    std::chrono::steady_clock::time_point t = std::chrono::steady_clock::now();
    void lap(const char *what) {
        if (!on) return;
        const auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "[nb200 trace] host %-24s %.3f s\n", what, std::chrono::duration<double>(now - t).count());
        t = now;
    }
};

struct Arena {                 // strings back to back: data + offsets (n + 1)
    std::string data;
    std::vector<int64_t> off{0};
    void add(const char *p, size_t n);
    size_t size() const { return off.size() - 1; }
    const char *ptr(size_t i) const { return data.data() + off[i]; }
    size_t len(size_t i) const { return (size_t)(off[i + 1] - off[i]); }
};

struct ReadSet {                // the pairs of the 10x one-pass route: corrected CB, raw UB, read 1, read 2
    Arena names, r1, r2, cb, ub;
};

void write_per_read_tsv(const std::string &out_path, const ReadSet &R, const nb200_read_result *res, const int32_t *feats,
                        int max_hits, const std::vector<std::string> &feature_names, int threads = 1);

// ---- fastq-to-bam (fastq2bam.cpp) -------------------------------------------------------------------
struct FqRec { uint64_t name, seq, qual; uint32_t name_len, len; };   // offsets into FastqQ::text
struct FastqQ { std::string text; std::vector<FqRec> recs; };
void load_fastq_qual(const std::string &path, FastqQ &F);
// process_pair's name check: r1.id.removesuffix('/1') == r2.id.removesuffix('/2')  (:152-156)
inline bool name_eq_stripped(const char *a, uint32_t la, const char *b, uint32_t lb) {
    if (la >= 2 && a[la - 2] == '/' && a[la - 1] == '1') la -= 2;
    if (lb >= 2 && b[lb - 2] == '/' && b[lb - 1] == '2') lb -= 2;
    return la == lb && std::char_traits<char>::compare(a, b, la) == 0;
}
void slice_barcodes(const FastqQ &A, const FastqQ &B, int cb_len, int umi_len, int threads, uint8_t *cb, uint8_t *qual,
                    uint8_t *eligible, nb200_cb_stats &st);
void write_10x_bam(const std::string &out_path, const FastqQ &A, const FastqQ &B, int cb_len, int umi_len, const int32_t *idx,
                   const uint8_t *status, const std::vector<std::string> &wl_entries, int threads, nb200_cb_stats &st);
void read_whitelist_lines(const std::string &path, std::vector<std::string> &lines);

// ---- report (report.cpp) --------------------------------------------------------------------------------
struct ReportRows {
    std::string text;                        // the TSV (string_views point into it while parsing)
    std::vector<std::string> feature_names;  // ascending; id = rank
    std::vector<std::string> cells;          // ascending; id = rank
    std::vector<uint64_t> key;               // cell id << 32 | umi id
    std::vector<uint32_t> off, ids;          // CSR of ascending feature ids per row
    std::vector<double> score;
};
bool parse_per_read_tsv(const std::string &path, ReportRows &R, int threads = 1);
void write_counts_tsv(const std::string &out_path, const nb200_counts *c, const std::vector<std::string> &feature_names,
                      const std::vector<std::string> &cells);

}  // namespace nb200
