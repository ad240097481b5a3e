// Streaming file pipeline behind nb200_align_files / nb200_align_files_multi (SURVEY.md §8a X2, X5; §8e):
//   reader + block-parallel inflate -> record walker (mate pairing) -> parse + 2-bit pack straight into page-locked slabs
//   -> one thread per GPU (two slabs in flight each, slab_api.hpp) -> TSV formatters -> ordered writer.
// Bounded memory: a fixed pool of slabs; every stage hands work on, nothing holds the whole file.
// Reference boundary: what the aligner process does between its argv and its exit code (nimble/__main__.py:177-196).
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/nimble_b200.h"

namespace nb200 {

struct FileJob {
    std::vector<std::string> inputs;      // one or two FASTQ(.gz), or one BAM
    std::vector<nb200_ctx *> ctxs;        // one context per GPU; empty = dry run (no device stage, reader statistics only)
    std::vector<int32_t> lib_ids;         // the same ids on every context (libraries loaded in the same order)
    std::vector<std::string> outputs;     // one per library (per-read TSV); empty in counts-only mode
    int host_threads = 1;
    // counts mode (nb200_align_files_counts): one counts TSV per library, the UMI stage on the device
    std::vector<std::string> counts_outputs;
    double umi_threshold = 0.05;
    int umi_flags = 0;                    // NB200_UMI_NO_THRESHOLD | NB200_UMI_CORRECT
    // 10x mode (nb200_fastq_to_counts, counts only): inputs = raw R1 and R2 FASTQ.  The pairs fastq-to-bam would write
    // go to the device as its BAM would: CB = R1[0, cb_len) corrected against the whitelist there, UB = R1[cb_len,
    // cb_len + umi_len), read 1 = the rest of R1, read 2 = R2.
    const std::vector<std::string> *whitelist = nullptr;   // the non-empty lines of the whitelist file; null = off
    int cb_len = 16, umi_len = 12;
};

struct FileStats {
    uint64_t n_reads = 0, paired = 0, has_tags = 0, bases1 = 0, bases2 = 0, checksum = 0, n_slabs = 0, called = 0;
    double seconds = 0.0;
    std::vector<uint64_t> counts3;        // counts mode: per library rows used, count rows written, UMIs dropped (+ UMIs corrected)
    nb200_cb_stats cb{};                  // 10x mode: fastq-to-bam's counters (cache_size 0: not computed by this route)
};

// throws IoError / std::exception
void run_file_pipeline(const FileJob &job, FileStats *stats);

}  // namespace nb200
