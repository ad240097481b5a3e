// Host file code outside the streaming pipeline: whole-file reads, the 10x one-pass route's per-read TSV, fastq-to-bam, report.
#pragma once
#include <chrono>
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
