// Host file code outside the streaming pipeline: whole-file reads, fastq-to-bam's BAM records, report.
#pragma once
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <exception>
#include <mutex>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "../../include/nimble_b200.h"

namespace nb200 {

struct IoError : std::runtime_error { using std::runtime_error::runtime_error; };

template <class F>
void parallel_for(int T, F &&fn) {                             // fn(t) on T threads
    if (T <= 1) { fn(0); return; }
    std::vector<std::thread> th;
    std::exception_ptr err;
    std::mutex em;
    for (int t = 0; t < T; t++)
        th.emplace_back([&, t] { try { fn(t); } catch (...) { std::lock_guard<std::mutex> g(em); if (!err) err = std::current_exception(); } });
    for (auto &x : th) x.join();
    if (err) std::rethrow_exception(err);
}

// ---- fastq-to-bam's records (fastq2bam.cpp; the 10x mode of the streaming pipeline writes them) ---------------------
// process_pair's name check: r1.id.removesuffix('/1') == r2.id.removesuffix('/2')  (:152-156)
inline bool name_eq_stripped(const char *a, uint32_t la, const char *b, uint32_t lb) {
    if (la >= 2 && a[la - 2] == '/' && a[la - 1] == '1') la -= 2;
    if (lb >= 2 && b[lb - 2] == '/' && b[lb - 1] == '2') lb -= 2;
    return la == lb && std::char_traits<char>::compare(a, b, la) == 0;
}
// one unaligned BAM record (:186-207) appended to out; qual is FASTQ text (phred + 33)
void bam_record(std::string &out, const char *name, uint32_t name_len, uint32_t flag, const char *seq, const char *qual,
                uint32_t len, const char *cb, uint32_t cb_len, const char *ub, uint32_t ub_len);
// raw BAM bytes -> BGZF blocks appended to out
void bgzf_blocks(const std::string &raw, std::string &out);
// the BGZF blocks of fastq-to-bam's header (:235-238), and the end-of-file block
std::string bam_header_bgzf();
extern const unsigned char kBgzfEof[28];
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
// cuts of text t at line ends ('\n') from `body` on: one piece per thread for a large body, one piece below 4 MB;
// returns pieces + 1 offsets, the last t.size()
std::vector<size_t> line_pieces(const std::string &t, size_t body, int threads);

// ---- report -s (summarize.cpp; DESIGN.md §2.13) -----------------------------------------------------------
enum SumKind : int { SUM_INT = 0, SUM_INT_AS_FLOAT, SUM_FLOAT, SUM_STRING };   // typed values of a column (frontend._infer_column)
struct SumColumn {
    int header_index = -1;
    SumKind kind = SUM_INT;
    std::vector<uint64_t> cell;        // per row: text offset << 24 | length (kSumAbsent: a pandas NA token)
    std::vector<uint64_t> key;         // per row with a cell: value identity, ascending in typed order, minus the smallest
    int bits = 1;                      // significant bits of the keys
};
constexpr uint64_t kSumAbsent = ~0ull;
struct SummaryTable {
    std::string text;
    uint64_t n_rows = 0;
    std::vector<SumColumn> cols;       // distinct header columns the summary reads
    int umi = 0;                       // index into cols of the `umi` column
    std::vector<int> out_cols;         // per requested column: index into cols
    std::vector<std::string> out_names;
};
// The column `name` (after renaming) is not in the header.
struct MissingColumn : std::runtime_error {
    std::string name;
    explicit MissingColumn(const std::string &n) : std::runtime_error("missing column: " + n), name(n) {}
};
void parse_summary_tsv(const std::string &path, const std::vector<std::string> &columns, SummaryTable &S, int threads);
// (umi rank, count, first row) per (UMI, value) pair of one column, in output order
struct SumRuns { std::vector<uint32_t> urank, count, first; };
void write_summary_tsv(const std::string &out_path, const SummaryTable &S, const std::vector<uint32_t> &umi_first,
                       const std::vector<SumRuns> &runs, int threads);
void write_counts_tsv(const std::string &out_path, const nb200_counts *c, const std::vector<std::string> &feature_names,
                      const std::vector<std::string> &cells);

}  // namespace nb200
