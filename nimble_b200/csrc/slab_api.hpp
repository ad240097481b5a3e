// GPU side of the streaming file pipeline (stream.cpp): a context runs up to two slabs (batches of parsed reads) at
// a time, each on its own "lane" of device buffers: H2D of slab k+1 and D2H of slab k-1 overlap the kernels of slab k.
#pragma once
#include <cstddef>
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/nimble_b200.h"

namespace nb200 {

constexpr int kFileLanes = 2;
// 10x mode, host key of a pair before correction: flags in the high half, the UMI (or kTenxNaUmi) in the low half
constexpr uint64_t kTenxLongRead = 1, kTenxLongName = 2;   // a read over 500 bases after the cut / a name over 254 bytes
constexpr uint32_t kTenxNaUmi = 0xFFFFFFFFu;               // (UMI ids stay below it: umi_code < 2^31, interned < 2^32 - 1)

// The calling thread becomes the one that drives this context's device (cudaSetDevice).
void lane_bind_thread(nb200_ctx *c);
// Enqueue one slab: copy the packed reads to the device, align against every library in lib_ids (the reads go up
// once), copy the per-read records / feature ids back into the caller's PINNED buffers (one pair per library).
// Asynchronous; throws std::exception on error.
// len1 / len2 (may be null): per library, the read lengths that library's kernels use instead of r1->len / r2->len
// (--trim keeps a per-library prefix of every read; the packed records are shared).
// out_res / out_feats may be null (counts only: no per-read results come back).
// key (counts mode, after lane_rows_begin): per read cell << 32 | umi or NB200_NO_BARCODE, PINNED; it goes up with the
// reads and every library's rows that count are appended to that library's row store on the device.
// cb (10x mode, after lane_cb_begin): the slab's raw cell barcodes; the device corrects them and copies each pair's
// correction back into cb's PINNED out buffers (read them after lane_wait).  With key (counts mode) key holds flags << 32 |
// umi on entry (kTenx*: umi kTenxNaUmi for a pandas-NA UMI) and the device fills the cell half (barcode.cuh:
// cb_key_kernel); a flagged read whose barcode is corrected makes lane_wait throw (the two-step route fails on exactly
// those pairs).  n_libs == 0 (fastq-to-bam): only the barcodes go up and are corrected, the reads are not uploaded.
// seq: the slab's place in the file (the cache rule's order).
struct CbSlab {
    const uint8_t *cb = nullptr, *qual = nullptr;  // in: n x cb_len raw bases / phred values
    int32_t *idx = nullptr;                        // out: whitelist line, or -1 (the device's own choice for a read with
    uint8_t *status = nullptr;                     //      several candidates: the host's resolve step decides those)
    uint8_t *multi = nullptr;                      // out: NB200_CB_* / 1 = several candidates
};
void lane_submit(nb200_ctx *c, int lane, const nb200_reads *r1, const nb200_reads *r2, const int32_t *lib_ids, int n_libs,
                 nb200_read_result *const *out_res, int32_t *const *out_feats, uint16_t *const *len1 = nullptr,
                 uint16_t *const *len2 = nullptr, const uint64_t *key = nullptr, const CbSlab *cb = nullptr, uint64_t seq = 0);
// --trim setting of a library (nb200_library_set_trim); false = none
bool lane_trim(nb200_ctx *c, int32_t lib_id, int *target, double *strictness);
// Block until the slab of this lane is done and its outputs are in the host buffers (re-runs it with a larger
// Smith-Waterman work list if that overflowed).
void lane_wait(nb200_ctx *c, int lane);
int lane_max_hits(nb200_ctx *c, int32_t lib_id);
const char *lane_feature_name(nb200_ctx *c, int32_t lib_id, uint32_t fid, uint32_t *len);
uint32_t lane_n_features(nb200_ctx *c, int32_t lib_id);
int lane_host_threads(nb200_ctx *c);
// page-lock / release an existing host range for every context of the process (cudaHostRegisterPortable); false = not pinned
bool lane_pin(void *p, size_t bytes);
void lane_unpin(void *p);

// ---- counts mode: the rows of the UMI stage never leave the device --------------------------------------------
// One row store per library and context: key u64, names per row u32, feature ids (CSR without offsets).  A slab
// appends one segment per library behind its calling kernels; segments are gathered in slab order at the end.
struct RowSeg {
    uint64_t seq = 0;            // slab sequence number (per-read TSV order)
    int ctx = 0;                 // index of the context in the call
    uint64_t row0 = 0, rows = 0, id0 = 0, ids = 0;   // where the segment lies in that context's store
    uint64_t called = 0;         // reads of the slab with a feature call (every read, not only rows that count)
};
// Empty the row stores of the libraries of this call and upload each library's "name is a pandas NA token" flags.
void lane_rows_begin(nb200_ctx *c, const int32_t *lib_ids, int n_libs);
// After lane_wait: the segment the lane's slab appended, per library (seq / ctx are the caller's to fill).
void lane_rows_segments(nb200_ctx *c, int lane, RowSeg *out);
// Gather the segments (in the order given) of library li from every context into ctxs[0], map the cell ids to ranks
// (cell_rank[id], so that cell order is byte order), run the UMI stage.  *counts is the context's table as
// nb200_umi_counts returns it; *rows = rows that reached the UMI stage.  Throws LimitError beyond 2^31 rows.
// tenx (fastq-to-counts, after lane_cb_resolve): cells are whitelist lines, provisional ones are decided first, and
// cell_rank is lane_cb_begin's rank (~0u: the row is dropped and not counted in *rows).  umi_flags: NB200_UMI_* (with
// NB200_UMI_CORRECT the UMIs are corrected after the cells are final).
void lane_rows_count(const std::vector<nb200_ctx *> &ctxs, int li, int32_t lib_id, const std::vector<RowSeg> &segs,
                     const std::vector<uint32_t> &cell_rank, double threshold, int umi_flags, nb200_counts *counts, uint64_t *rows,
                     bool tenx = false);

// ---- 10x mode: cell barcodes corrected slab by slab, the correction cache over the whole call ---------------------
// Upload the whitelist table to every context and empty their logs of reads with several candidates.  rank[i] = rank
// of whitelist line i among the distinct lines in byte order, ~0u for a line that can never match or is a pandas NA
// token (report drops such a cell); cells[rank] = the line.  cache_size: also keep what lane_cb_cache_size counts.
void lane_cb_begin(const std::vector<nb200_ctx *> &ctxs, const std::vector<std::string> &whitelist, int cb_len,
                   std::vector<uint32_t> *rank, std::vector<std::string> *cells, bool cache_size = false);
// After lane_wait: the slab's perfect matches, corrections, no-corrections, exact misses, multi-candidate reads, probes.
void lane_cb_counters(nb200_ctx *c, int lane, uint64_t *out6);
// After the last slab: the first read (in file order) of each raw barcode among the logged ones decides for all of them
// (the reference's correction_cache, DESIGN.md §2.8); the decisions stay on ctxs[0] for lane_rows_count.
void lane_cb_resolve(const std::vector<nb200_ctx *> &ctxs);
// After the last slab (lane_cb_begin with cache_size): distinct raw barcodes of the call made of ACGTN only = whitelist
// entries hit exactly on any context + distinct raw barcodes among the exact misses of every context.
uint64_t lane_cb_cache_size(const std::vector<nb200_ctx *> &ctxs);
// Free the whitelist tables and logs of the call.
void lane_cb_end(const std::vector<nb200_ctx *> &ctxs);

}  // namespace nb200
