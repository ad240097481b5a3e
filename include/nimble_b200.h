/* nimble_b200 — C ABI of the B200-native replacement for nimble's read-assignment hot path.
 *
 * The reference has no FFI for this path: nimble/__main__.py:153-211 (`align`) builds an argv
 * (`--input F.. -c N --strand_filter S {-r LIB.json -o OUT}.. [-t TRIM]`, :177-192), execs the
 * external `nimble/aligner` binary (:195-196) and forwards its exit code (:198,211); the
 * per-read TSV it writes is consumed by `report` (nimble/__main__.py:213-293).  The entry
 * points below are what a ctypes binding placed in `align()` / `report()` calls instead of
 * that exec (see INTEGRATION.md for the stub); every one cites the reference site it replaces.
 *
 * Conventions: plain pointers and sizes only; every function returns int32 0 on success or a
 * negative NB200_E* code, with text available from nb200_last_error().  A context is not
 * re-entrant.  There is NO CPU fallback: without a CUDA device nb200_create fails with
 * NB200_ENODEVICE.
 */
#ifndef NIMBLE_B200_H
#define NIMBLE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NB200_OK 0
#define NB200_EINVAL (-1)     /* bad argument / malformed library JSON / read too long         */
#define NB200_ENODEVICE (-2)  /* no CUDA device (there is no CPU path)                          */
#define NB200_ECUDA (-3)      /* CUDA runtime error                                             */
#define NB200_EIO (-4)        /* file could not be read / written                               */
#define NB200_ELIMIT (-5)     /* library exceeds a documented limit (see DESIGN.md §5)          */

#define NB200_MAX_READ_LEN 500
#define NB200_NO_BARCODE UINT64_MAX

/* Flags word of the counting entries (the `int32_t disable_thresholding` parameter of nb200_umi_counts,
 * nb200_report_file, nb200_align_files_counts(_multi), nb200_fastq_to_counts(_multi); 0 and 1 keep their meaning):
 * NB200_UMI_NO_THRESHOLD skips the per-UMI proportional thresholding; NB200_UMI_CORRECT merges, per cell, each UMI into
 * its best-supported one-substitution neighbour before the UMI stage (DESIGN.md §2.12).  With NB200_UMI_CORRECT, out3
 * holds 4 values per library: the 3 documented at each entry, then the number of (cell, UMI) keys corrected.  Other bits:
 * NB200_EINVAL.  nb200_align and nb200_align_resident refuse NB200_UMI_CORRECT (their keys are caller-assigned ids). */
#define NB200_UMI_NO_THRESHOLD 1
#define NB200_UMI_CORRECT 2

/* strand filter: the reference forwards `--strand_filter` verbatim (nimble/__main__.py:180,399) */
enum { NB200_UNSTRANDED = 0, NB200_FIVEPRIME = 1, NB200_THREEPRIME = 2, NB200_STRAND_NONE = 3 };

/* Per-library alignment config = element 0 of the library JSON (nimble/types.py:12-25). */
typedef struct nb200_config {
    int32_t k;                        /* k-mer length, 4..32 (not in the JSON; engine parameter) */
    int32_t score_threshold;          /* types.py:12 */
    int32_t score_filter;             /* types.py:13 */
    double score_percent;             /* types.py:14 */
    int32_t num_mismatches;           /* types.py:15 */
    int32_t discard_multiple_matches; /* types.py:16 */
    int32_t intersect_level;          /* types.py:17 */
    int32_t discard_multi_hits;       /* types.py:19 */
    int32_t require_valid_pair;       /* types.py:20 */
    int32_t max_hits_to_report;       /* types.py:23 */
    int32_t strand_filter;            /* NB200_UNSTRANDED.. (CLI level, __main__.py:399) */
    int32_t pad_;
} nb200_config;

/* One batch of reads, 2-bit packed by nb200_pack_reads (north-star subsystem 2).
 * Record i lives at packed + i*stride: [seq: words u64][nmask: words u32], little-endian,
 * base j at bits [2(j%32), 2(j%32)+2) of seq word j/32, A=0 C=1 G=2 T=3, nmask bit j set when
 * base j is not ACGT.  words = ceil(max_len/32); stride = 12*words rounded up to 16.
 *
 * Compact wire form (nb200_pack_reads_compact; stride == 8*words): the records hold the seq words only and
 * the few reads with a non-ACGT base are listed in a side table — n_idx[j] = read index (ascending),
 * n_mask[j*words ..] = its nmask words.  24 B instead of 48 B per 90-base read cross PCIe; the device
 * expands the records to the full form (expand_reads_kernel) before the first kernel reads them. */
typedef struct nb200_reads {
    const uint8_t *packed;
    const uint16_t *len;      /* bases per read */
    uint64_t n;
    uint32_t stride;
    uint32_t words;
    const uint32_t *n_idx;    /* compact form only (else NULL / 0) */
    const uint32_t *n_mask;
    uint64_t n_with_n;
} nb200_reads;

/* Per-read outcome (what the aligner writes as one TSV row; nimble/__main__.py:237-241 consumes
 * nimble_features / nimble_score / r1_CB / r1_UB).  Index order: r1 fwd, r1 rc, r2 fwd, r2 rc. */
typedef struct nb200_read_result {
    uint16_t score[4];   /* alignment score in bp */
    uint16_t n_hits[4];  /* index k-mers hit */
    uint16_t n_cand[4];  /* equivalence-class size after refinement (saturates at 65535) */
    uint8_t edits[4];
    uint8_t status[4];   /* 0 none 1 pass 2 no-match 3 empty-class 4 score 5 percent 6 multiple */
    uint8_t reason;      /* 0 called 1 no-pass 2 not-valid-pair 3 force-intersect 4 score-filter 5 multi-hits 6 max-hits */
    uint8_t config;      /* 0 F 1 R 2 FF 3 RR, 255 none */
    uint8_t n_feat;
    uint8_t n_sw;        /* orientations that needed Smith-Waterman */
    uint32_t pair_score;
} nb200_read_result;

/* Count table = the rows of the counts TSV `feature<TAB>count<TAB>cell_barcode`
 * (nimble/__main__.py:289-293), already in the reference's output order
 * (ascending cell, then ascending comma-joined feature string).  Owned by the context, valid
 * until the next call on it. */
typedef struct nb200_counts {
    uint64_t n_rows;
    const uint32_t *cell;       /* upper 32 bits of the read key */
    const uint32_t *count;      /* UMIs */
    const uint32_t *feat_off;   /* n_rows + 1 */
    const uint32_t *feat_ids;   /* feature ids; names via nb200_feature_name */
    uint64_t dropped_empty;     /* "Dropped N UMIs due to empty intersections" (__main__.py:279) */
    uint64_t n_called;          /* reads with a feature call */
    uint64_t n_umis;            /* (cell, umi) groups seen */
} nb200_counts;

/* Device-side timings of the last nb200_align_* call (CUDA events, milliseconds).  The three stage times are
 * summed over the batches of the call, each measured on the stream the stage runs on: with batch pipelining on
 * (nb200_set_overlap, default) stages of neighbouring batches overlap and the sum exceeds total_ms. */
typedef struct nb200_timing {
    float total_ms;     /* first H2D (or first kernel) -> count table ready on the host        */
    float probe_ms;     /* k-mer extraction + hash probe + class intersection + direct calling */
    float sw_ms;        /* window fingerprint + dedupe + banded Smith-Waterman kernels         */
    float call_ms;      /* score / strand / pair filter + feature calling of the aligned reads */
    float agg_ms;       /* radix sorts + per-UMI threshold/intersect + run-length count + table D2H */
    float h2d_ms;
    uint64_t probes;    /* hash-table lookups issued (device counter; 0 unless nb200_set_stats(1)) */
    uint64_t probe_slots; /* 32-byte buckets (L2 sectors) read for them               */
    uint64_t sw_pairs;  /* (read orientation, candidate) pairs aligned (distinct windows) */
    uint64_t sw_cells;  /* DP cells = sum L*(2w+1)                                      */
    uint64_t launches;  /* kernels launched inside the call (ours + CUB)               */
    uint64_t h2d_bytes, d2h_bytes;
    uint64_t sw_items;  /* candidate pairs before identical band windows were merged   */
    float probe_kernel_ms; /* the probe kernels alone (part of probe_ms, which also covers the calling kernels that follow it) */
    float pad_;
    uint64_t probe_warp_reads; /* single-end reads the thread-per-read probe left to the warp-per-read probe */
} nb200_timing;

typedef struct nb200_ctx nb200_ctx;

/* lifecycle — replaces locating/downloading the binary (nimble/__main__.py:154-166) */
int32_t nb200_create(int32_t device, int32_t host_threads, nb200_ctx **out);
void nb200_destroy(nb200_ctx *ctx);
const char *nb200_last_error(const nb200_ctx *ctx);   /* NULL ctx -> last create error */
const char *nb200_version(void);

/* `-r LIB.json` (nimble/__main__.py:182-189): parse [config, data] (nimble/__main__.py:64-65,
 * nimble/types.py:10-32), build the k-mer -> equivalence-class index and upload it.
 * strand_filter: "unstranded" | "fiveprime" | "threeprime" | "none".
 * The path may also name an index file written by nb200_index_write (told apart by its magic bytes, not its
 * extension): it is loaded without a build and each device checks its copy of the image (a damaged file is
 * NB200_EINVAL, nothing is registered).  k <= 0: the index's own k (20 for a JSON); any other k that differs from an
 * index's k is NB200_EINVAL.  So every entry that takes library paths (the *_multi calls too) takes index files. */
int32_t nb200_load_library(nb200_ctx *ctx, const char *json_path, const char *strand_filter, int32_t k,
                           int32_t *lib_id);
/* same, from memory: names/sequences/feature names per reference + explicit config */
int32_t nb200_load_library_mem(nb200_ctx *ctx, int32_t n_refs, const char *const *names,
                               const char *const *seqs, const char *const *features,
                               const nb200_config *cfg, int32_t *lib_id);
int32_t nb200_library_config(const nb200_ctx *ctx, int32_t lib_id, nb200_config *out);
int32_t nb200_library_set_config(nb200_ctx *ctx, int32_t lib_id, const nb200_config *cfg); /* k is fixed */
/* `-t <TARGET_LENGTH>:<STRICTNESS>` (nimble/__main__.py:191-192,400; defaults nimble/types.py:24-25), one entry per
 * library: reads of the FILE-level calls (nb200_align_files*) are quality-trimmed for this library before alignment —
 * the prefix that maximises the MaxInfo criterion (DESIGN.md §2.9) is kept; input without qualities is not trimmed.
 * target_length < 0 switches it off (default).  nb200_align with caller buffers is unaffected (the caller owns len[]). */
int32_t nb200_library_set_trim(nb200_ctx *ctx, int32_t lib_id, int32_t target_length, double strictness);
/* the criterion itself (host only, no context): bases to keep of a read with these qualities (5' -> 3') */
uint32_t nb200_trim_maxinfo(const uint8_t *qual, uint32_t n, int32_t phred_offset, int32_t target_length, double strictness);
int32_t nb200_library_info(const nb200_ctx *ctx, int32_t lib_id, int64_t *n_refs, int64_t *n_features,
                           int64_t *n_kmers, int64_t *n_classes, int64_t *table_bytes);
const char *nb200_feature_name(const nb200_ctx *ctx, int32_t lib_id, uint32_t feature_id);
/* host-only dry run of nb200_load_library (no CUDA call): out6 = n_refs, n_features, n_kmers,
 * n_classes, n_slots, identity_features.  Errors via nb200_last_error(NULL). */
int32_t nb200_host_index_stats(const char *json_path, const char *strand_filter, int32_t k, int64_t *out6);
/* host-only (no CUDA call, runs on a machine without a GPU): build the index of `json_path` at k (<= 0: 20) and write
 * it to out_path (via out_path.tmp, then rename) as an index file (DESIGN.md §4) that nb200_load_library reads in
 * place of the JSON.  host_threads <= 0: all cores.  Errors via nb200_last_error(NULL). */
int32_t nb200_index_write(const char *json_path, int32_t k, int32_t host_threads, const char *out_path);
/* host-only: header of an index file.  out9 = format version, k, n_refs, n_features, n_kmers, n_classes, n_slots,
 * identity_features (as nb200_host_index_stats), device image bytes.  The header and host sections are always checked;
 * verify = 1 also checks the image's checksum and looks every valid k-mer of every reference up in the image read back
 * (it must find a class that holds that reference).  A damaged or foreign file: NB200_EINVAL with the reason. */
int32_t nb200_index_info(const char *path, int32_t verify, int64_t *out9);

/* test hook (host only): the one-substitution neighbours of UMI code `code` as the correction kernel visits them
 * (codes and byte-order values, see nb200_umis_corrected); returns their number (<= 52), -1 for a value that is not a
 * code.  out_code / out_value hold 52 entries. */
int32_t nb200_umi_neighbours(uint32_t code, uint32_t *out_code, uint32_t *out_value);

/* test hook (host only): the raw-DEFLATE decoder the BGZF reader tries before zlib (csrc/fast_inflate.hpp).
 * 1 = the stream decoded into exactly out_len bytes, 0 = declined (the reader then uses zlib). */
int32_t nb200_fast_inflate(const uint8_t *in, uint64_t in_len, uint8_t *out, uint64_t out_len);

/* host-only dry run of the file reader behind nb200_align_files (no CUDA call): FASTQ(.gz) x1-2 or BAM.
 * out6 = n_reads, paired, has_tags, total read-1 bases, total read-2 bases, FNV-1a checksum over
 * (name, r1[, r2][, CB, UB]) of every read in order.  Errors via nb200_last_error(NULL). */
int32_t nb200_host_ingest_stats(const char *const *inputs, int32_t n_inputs, int32_t threads, uint64_t *out6);

/* read ingest (north-star subsystem 2): ASCII -> packed records, host threads.
 * bases: concatenated ASCII, off[n+1].  out must hold n*stride bytes, out_len n entries. */
int32_t nb200_pack_layout(uint32_t max_len, uint32_t *words, uint32_t *stride);
int32_t nb200_pack_reads(nb200_ctx *ctx, const char *bases, const int64_t *off, uint64_t n,
                         uint32_t words, uint32_t stride, uint8_t *out, uint16_t *out_len);
/* compact wire form (see nb200_reads): out holds n*8*words bytes; reads with a non-ACGT base go to the side table
 * (out_n_idx: cap entries, out_n_mask: cap*words).  *n_with_n = entries needed; NB200_ELIMIT when cap is too small
 * (nothing but *n_with_n is valid then: call again with larger tables). */
int32_t nb200_pack_reads_compact(nb200_ctx *ctx, const char *bases, const int64_t *off, uint64_t n, uint32_t words,
                                 uint8_t *out, uint16_t *out_len, uint32_t *out_n_idx, uint32_t *out_n_mask,
                                 uint64_t cap, uint64_t *n_with_n);
/* barcode strings (fixed width <= 16 / <= 16, ACGT) -> key = cb << 32 | ub; non-ACGT -> NB200_NO_BARCODE */
int32_t nb200_pack_barcodes(const char *cb, uint32_t cb_len, const char *ub, uint32_t ub_len, uint64_t n,
                            uint64_t *out_key);
void *nb200_alloc_pinned(size_t bytes);
void nb200_free_pinned(void *p);

/* THE hot path — replaces Popen([aligner] + argv).wait() (nimble/__main__.py:195-196) followed by
 * report() (nimble/__main__.py:254-293) for one library.
 * r2 may be NULL (single-end).  key[i] = cell << 32 | umi (NB200_NO_BARCODE = no CB/UB tag; such
 * reads are aligned but not counted, like report's dropna at __main__.py:244); key == NULL means
 * bulk data: rows are counted per feature set with cell = 0.
 * Host buffers in, count table out; the H2D copies run ahead of the kernels in ramped batches on a copy stream.
 * results / feats (n * max_hits_to_report, -1 padded) may be NULL when only counts are wanted. */
int32_t nb200_align(nb200_ctx *ctx, int32_t lib_id, const nb200_reads *r1, const nb200_reads *r2,
                    const uint64_t *key, double umi_threshold, int32_t disable_thresholding,
                    nb200_read_result *results, int32_t *feats, nb200_counts *counts);

/* File-level form of the same call — exactly what the aligner process does for
 * `--input F.. {-r LIB -o OUT}..` (nimble/__main__.py:177-196): FASTQ(.gz) x1-2 or BAM in (native
 * BGZF reader, CB/UB/UR/GN tags), one per-read TSV per library out (columns nimble_features,
 * nimble_score, r1_CB, r1_UB, ... consumed at nimble/__main__.py:237-241; `features<TAB>count` with
 * a header for FASTQ input, nimble/parse.py:39-57).  OUT ending in .gz is gzip-compressed (one gzip member per slab
 * of reads); files are written to OUT.tmp and renamed.
 * Streaming: reader / block-parallel inflate -> record parse + 2-bit pack into pinned slabs -> cudaMemcpyAsync ->
 * kernels -> per-read results back into pinned memory -> TSV formatters -> ordered writer, all overlapped; host memory
 * is bounded by the slab pool, not by the file size.  Paired BAM records are matched by name at any distance; rows of
 * pairs whose mates are not adjacent come out where the second mate was read. */
int32_t nb200_align_files(nb200_ctx *ctx, const char *const *inputs, int32_t n_inputs, const int32_t *lib_ids,
                          const char *const *outputs, int32_t n_libs);

/* nb200_align_files over several GPUs of one node from ONE process (SURVEY.md §8e; no context needed: one is created
 * per device for the duration of the call).  Every library is loaded on every device (index replicated); the reader
 * hands slabs of reads to whichever GPU has a free lane and the writer restores input order, so the outputs are
 * byte-identical to a one-GPU run.  trim: the `-t` value ("L:S[,L:S...]", one entry per library) or NULL / "".
 * err (may be NULL) receives the message on failure; stats4 (may be NULL) = reads,
 * seconds (pipeline only, libraries loaded), reads with a feature call, slabs. */
int32_t nb200_align_files_multi(const int32_t *devices, int32_t n_devices, int32_t host_threads, const char *const *inputs, int32_t n_inputs,
                                const char *const *library_json, int32_t n_libs, const char *strand_filter, int32_t k,
                                const char *const *outputs, const char *trim, char *err, size_t err_cap, double *stats4);

/* `align` (nimble/__main__.py:153-211) followed by `report` (nimble/__main__.py:254-293) in one streaming pass: BAM with
 * CB / UB tags in, one counts TSV `feature<TAB>count<TAB>cell_barcode` per library out, byte-identical to
 * nb200_align_files + nb200_report_file on the same input.  The called rows never leave the device: each slab appends the
 * rows report would keep (a call, valid CB and UB, not one feature named like a pandas NA token) to a row store behind its
 * calling kernels; after the last slab the rows are gathered in per-read TSV order, cells ranked by CB bytes, and the
 * UMI stage (nb200_umi_counts, score 1 per row) runs on them.
 * per_read_outputs may be NULL (no per-read TSV); otherwise the per-read TSVs are written in the same pass, identical to
 * nb200_align_files'.  counts_outputs: one path per library.
 * out3 (may be NULL): per library 3 values = rows used, count rows written, UMIs dropped (as nb200_report_file).
 * FASTQ input or a BAM without any CB / UB tag fails (NB200_EINVAL); so does a library feature name containing
 * ',', TAB, LF or CR (the per-read TSV cannot carry it).  More than 2^31 rows of one library: NB200_ELIMIT. */
int32_t nb200_align_files_counts(nb200_ctx *ctx, const char *const *inputs, int32_t n_inputs, const int32_t *lib_ids,
                                 const char *const *per_read_outputs, const char *const *counts_outputs, int32_t n_libs,
                                 double umi_threshold, int32_t disable_thresholding, uint64_t *out3);
/* The same over several GPUs (as nb200_align_files_multi): slabs go to whichever device has a free lane, each device
 * keeps its own row store, the cell dictionary is shared, and the rows are gathered on devices[0] (cudaMemcpyPeerAsync,
 * peer access where the devices allow it).  devices may repeat an index ({0, 0}: two contexts on one GPU).  Outputs are
 * byte-identical to a one-GPU run. */
int32_t nb200_align_files_counts_multi(const int32_t *devices, int32_t n_devices, int32_t host_threads,
                                       const char *const *inputs, int32_t n_inputs, const char *const *library_json,
                                       int32_t n_libs, const char *strand_filter, int32_t k, const char *trim,
                                       const char *const *per_read_outputs, const char *const *counts_outputs,
                                       double umi_threshold, int32_t disable_thresholding,
                                       uint64_t *out3, char *err, size_t err_cap, double *stats4);

/* Same computation with inputs already resident in HBM: upload once, then time repeated passes. */
int32_t nb200_upload(nb200_ctx *ctx, const nb200_reads *r1, const nb200_reads *r2, const uint64_t *key);
int32_t nb200_align_resident(nb200_ctx *ctx, int32_t lib_id, double umi_threshold,
                             int32_t disable_thresholding, nb200_counts *counts);
int32_t nb200_fetch_results(nb200_ctx *ctx, nb200_read_result *results, int32_t *feats);
/* Device copies of the last count table (same layout as nb200_counts: cell[n_rows], count[n_rows],
 * feat_off[n_rows + 1], feat_ids[n_ids]) so that the multi-GPU gather of the per-shard tables can run
 * device to device over NVLink (SURVEY.md §8e).  Valid until the next call on the context. */
int32_t nb200_counts_device(const nb200_ctx *ctx, uint64_t *n_rows, uint64_t *n_ids, const uint32_t **cell,
                            const uint32_t **count, const uint32_t **feat_off, const uint32_t **feat_ids);

/* report() on its own (nimble/__main__.py:254-293): rows (key, feature list, score) -> counts.
 * feat_ids ascending per row (duplicates allowed), off[n+1]; score NULL = 1.0 per row. */
int32_t nb200_umi_counts(nb200_ctx *ctx, int32_t lib_id, uint64_t n_rows, const uint64_t *key,
                         const uint32_t *off, const uint32_t *feat_ids, const double *score,
                         double umi_threshold, int32_t disable_thresholding, nb200_counts *counts);
/* (cell, UMI) keys corrected by the last UMI stage run on the context (0 without NB200_UMI_CORRECT).  With
 * NB200_UMI_CORRECT, nb200_umi_counts reads the UMI as the low half of the key: 1 ..= 1525878905 is the bijective base-5
 * code of an ACGTN string of 1..13 bases (A C G T N = digits 1..5, last base least significant); any other value is an
 * id that is never corrected. */
int32_t nb200_umis_corrected(const nb200_ctx *ctx, uint64_t *out);
/* report() file to file (nimble/__main__.py:254-293): per-read TSV (.gz or plain; columns nimble_features,
 * nimble_score, r1_CB, r1_UB) -> `feature<TAB>count<TAB>cell_barcode` without header, rows in the
 * reference's order.  Rows with a missing cell (pandas' NaN markers) are dropped (:244-245); an input
 * without usable rows gives an empty output (write_empty_df, :299-302).  out3 = rows used, count rows
 * written, UMIs dropped for an empty intersection (:279).  Native parser and writer, UMI stage on the GPU. */
int32_t nb200_report_file(nb200_ctx *ctx, const char *in_tsv, const char *out_tsv, double umi_threshold,
                          int32_t disable_thresholding, uint64_t *out3);
/* feature dictionary for nb200_umi_counts when rows come from a TSV: names sorted ascending */
int32_t nb200_load_feature_names(nb200_ctx *ctx, int32_t n, const char *const *names, int32_t *lib_id);

/* ---- fastq-to-bam: 10x cell-barcode correction (nimble/fastq_barcode_processor.py) ----------------
 * Replaces build_hamming_index (:17-36) + correct_cell_barcode (:73-128): exact whitelist match,
 * else the whitelist entries one substitution away, the one whose differing base has the lowest
 * quality wins (ascending string order on equal quality); the first read carrying a raw barcode
 * decides for all later reads with the same raw barcode (the reference's correction_cache). */
enum { NB200_CB_SKIPPED = 0, NB200_CB_PERFECT = 1, NB200_CB_CORRECTED = 2, NB200_CB_NONE = 3 };

/* The counters fastq_to_bam_with_barcodes prints (:284-309) + device timings of the last call. */
typedef struct nb200_cb_stats {
    uint64_t total_pairs, written_pairs;
    uint64_t cb_perfect_match, cb_corrected, cb_no_correction;
    uint64_t name_mismatch, too_short, no_remaining_seq;
    uint64_t cache_size;        /* distinct raw barcodes seen ("Correction cache size") */
    uint64_t n_exact_miss;      /* reads that needed the Hamming-1 search */
    uint64_t n_multi;           /* reads with several candidates (quality decides)  */
    uint64_t probes;            /* whitelist slots read */
    uint64_t launches;
    uint64_t h2d_bytes, d2h_bytes;
    float kernel_ms;            /* exact + Hamming + cache + statistics kernels, inputs resident (CUDA events) */
    float total_ms;             /* first H2D -> results on the host              */
} nb200_cb_stats;

/* load_cb_whitelist (:38-71): one barcode per line, .gz or plain; lines are stripped, empty lines
 * skipped.  Entry index = line order among the non-empty lines (first occurrence for duplicates).
 * Entries whose length is not cb_len can never match and are ignored; an entry of length cb_len
 * with a byte outside ACGTN is NB200_EINVAL.  cb_len <= 21. */
int32_t nb200_load_whitelist(nb200_ctx *ctx, const char *path, int32_t cb_len, int32_t *wl_id);
/* same from memory: n entries of cb_len bytes back to back */
int32_t nb200_load_whitelist_mem(nb200_ctx *ctx, const char *entries, uint64_t n, int32_t cb_len, int32_t *wl_id);
int32_t nb200_whitelist_info(const nb200_ctx *ctx, int32_t wl_id, int64_t *n_entries, int64_t *n_unique,
                             int64_t *table_bytes, int32_t *cb_len);
const char *nb200_whitelist_entry(const nb200_ctx *ctx, int32_t wl_id, uint32_t idx);

/* correct_cell_barcode over a batch, in file order.  cb, qual: n x cb_len bytes (ASCII bases /
 * phred values, any monotone encoding); eligible: n bytes or NULL (reads that fail process_pair's
 * earlier checks, :152-165, never reach the cache).  out_idx: whitelist entry index or -1;
 * out_status: NB200_CB_*.  stats may be NULL. */
int32_t nb200_correct_barcodes(nb200_ctx *ctx, int32_t wl_id, const char *cb, const uint8_t *qual,
                               const uint8_t *eligible, uint64_t n, int32_t *out_idx, uint8_t *out_status,
                               nb200_cb_stats *stats);
/* same with the batch already resident in HBM (device-timed benchmark arm) */
int32_t nb200_cb_upload(nb200_ctx *ctx, int32_t cb_len, const char *cb, const uint8_t *qual, const uint8_t *eligible,
                        uint64_t n);
int32_t nb200_correct_barcodes_resident(nb200_ctx *ctx, int32_t wl_id, int32_t *out_idx, uint8_t *out_status,
                                        nb200_cb_stats *stats);

/* `nimble fastq-to-bam` (fastq_to_bam_with_barcodes, :212-316): paired 10x FASTQ(.gz) + whitelist ->
 * unaligned BAM with CB (corrected) / UB (raw) tags, flags 77 / 141, read 1 = R1 minus barcode+UMI.
 * Pairs are written in file order. */
int32_t nb200_fastq_to_bam(nb200_ctx *ctx, const char *r1_fastq, const char *r2_fastq, const char *whitelist_path,
                           const char *output_bam, int32_t cb_len, int32_t umi_len, nb200_cb_stats *stats);
/* fastq-to-bam followed by align, without the intermediate BAM (SURVEY.md §8f rank 2): exactly the pairs
 * nb200_fastq_to_bam would write are aligned as nb200_align_files would align that BAM; one per-read TSV
 * per library.  Not a reference entry point: the reference needs both commands and the file between them. */
int32_t nb200_align_10x_fastq(nb200_ctx *ctx, const char *r1_fastq, const char *r2_fastq, const char *whitelist_path,
                              int32_t cb_len, int32_t umi_len, const int32_t *lib_ids, const char *const *outputs,
                              int32_t n_libs, nb200_cb_stats *stats);

/* fastq-to-bam followed by align --counts (nb200_align_files_counts) on its BAM, in one streaming pass and without the
 * BAM: raw 10x R1 / R2 FASTQ(.gz) + whitelist in, one counts TSV per library out, byte-identical to the two steps.  Pairs
 * are zipped in file order and stop at the shorter file; process_pair's rules pick the pairs that reach the correction;
 * each slab's barcodes are corrected on the device, and the first read (in file order) with a raw barcode that has
 * several candidates decides for every later read with it, across slabs and devices.  Memory is bounded by the slab pool.
 * --trim (nb200_library_set_trim) sees the qualities the BAM would hold.  out3 as nb200_align_files_counts; stats (may be
 * NULL): nb200_fastq_to_bam's counters, summed per slab; cache_size is not computed by this route and is 0.  It fails
 * where the two steps fail: a pair whose barcode is corrected (so fastq-to-bam writes it) with a read over 500 bases after
 * the barcode and UMI are cut off, or with a name over 254 bytes. */
int32_t nb200_fastq_to_counts(nb200_ctx *ctx, const char *r1_fastq, const char *r2_fastq, const char *whitelist_path,
                              int32_t cb_len, int32_t umi_len, const int32_t *lib_ids, const char *const *counts_outputs,
                              int32_t n_libs, double umi_threshold, int32_t disable_thresholding, uint64_t *out3,
                              nb200_cb_stats *stats);
/* The same over several GPUs, as nb200_align_files_counts_multi (devices may repeat an index); byte-identical to a
 * one-GPU run. */
int32_t nb200_fastq_to_counts_multi(const int32_t *devices, int32_t n_devices, int32_t host_threads, const char *r1_fastq,
                                    const char *r2_fastq, const char *whitelist_path, int32_t cb_len, int32_t umi_len,
                                    const char *const *library_json, int32_t n_libs, const char *strand_filter, int32_t k,
                                    const char *trim, const char *const *counts_outputs, double umi_threshold,
                                    int32_t disable_thresholding, uint64_t *out3, nb200_cb_stats *stats, char *err, size_t err_cap,
                                    double *stats4);

int32_t nb200_last_timing(const nb200_ctx *ctx, nb200_timing *out);
/* Batch pipelining (default on): batch k's fingerprint / Smith-Waterman / deferred-call kernels run on a
 * high-priority stream beside batch k+1's probe kernel.  Off = one stream, kernels back to back: the stage
 * times of nb200_timing then add up to total_ms (used to time each kernel alone for the roofline). */
int32_t nb200_set_overlap(nb200_ctx *ctx, int32_t on);

/* Deferred fetch (multi-GPU: SURVEY.md §8e): with it on, nb200_align / nb200_align_resident return as soon as the count table
 * is complete ON THE DEVICE (counts->n_rows set, host pointers NULL; nb200_counts_device gives the device arrays), so that
 * the caller can start the NVLink gather of the per-GPU tables and run nb200_fetch_counts — the D2H copy into the
 * context's pinned table — beside it instead of before it. */
int32_t nb200_set_defer_fetch(nb200_ctx *ctx, int32_t on);
int32_t nb200_fetch_counts_start(nb200_ctx *ctx);                      /* enqueue the copies and return (optional) */
int32_t nb200_fetch_counts(nb200_ctx *ctx, nb200_counts *counts);      /* start them if need be, wait, hand out the host table */

/* Device counters of the probe (nb200_timing.probes / probe_slots: table lookups issued, 32 B sectors read).  Off by
 * default: the two warp reductions and atomics per read cost instruction-issue slots in the kernel that is bound by them.
 * bench.py turns them on for the untimed passes its roofline block is computed from. */
int32_t nb200_set_stats(nb200_ctx *ctx, int32_t on);

/* Measurement helper (bench.py): achieved bandwidth of independent uniformly random 32 B-sector
 * gathers over a `bytes` buffer — the measured roofline of the hash probe (SURVEY.md §8d). */
int32_t nb200_bench_random_access(nb200_ctx *ctx, uint64_t bytes, uint32_t iters, double *gbytes_per_s,
                                  double *gloads_per_s);

/* Measurement helper (bench.py): integer-pipe ceilings of the Smith-Waterman kernel, register-only loops at full
 * occupancy.  dpx_ginst_per_s: thread-level DPX instructions per second (VIADDMNMX.S16x2.RELU and VIMNMX3.S16x2
 * issued 2 : 1 as in the kernel); row_gcups: cell updates per second of the kernel's own row recurrence without
 * any memory access (two alignments per thread in the s16 halves). */
int32_t nb200_bench_dpx_peak(nb200_ctx *ctx, uint32_t iters, double *dpx_ginst_per_s, double *row_gcups);

#ifdef __cplusplus
}
#endif
#endif
