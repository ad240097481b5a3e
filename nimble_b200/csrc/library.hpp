// Host-side library model: nimble's `[config, data]` JSON -> features -> k-mer index images that
// engine.cu uploads verbatim into HBM.  Reference surface: nimble/types.py:10-32 (schema),
// nimble/__main__.py:64-65 (file layout), nimble/__main__.py:182-189 (`-r LIB.json`).
#pragma once
#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/nimble_b200.h"

namespace nb200 {

constexpr uint32_t kEmptyClass = 0xFFFFFFFFu;
constexpr uint32_t kRefPad = 640;        // invalid bases before/after every reference (>= 500 + band + 64)
                                          // (a 500-base read may overhang a reference by 480: test_long_reads_gpu.py::test_reference_overhangs)
constexpr uint32_t kMaxRefs = 65535u * 32u;        // class words are indexed with 16 bits, 0xFFFF = no word

// k-mer table: bucketed cuckoo hashing keyed by the CANONICAL k-mer.  Entry = 16 B; bucket = 2 entries = 32 B =
// one L2 sector (a change to Entry, DualRec or ClassRec must bump kIndexVersion).  A key lives in its first bucket b1 or in its second bucket b2 (two independent 32-bit halves of
// hash_kmer, range-reduced by multiply-high); the SPILL bit of a bucket says "some key whose b1 is this bucket
// lives in its b2", so a lookup is one sector load plus, for the few flagged buckets, a second one - straight-line,
// no probe loop.  One entry answers both read orientations.
struct Entry {
    uint64_t key;        // min(x, revcomp x); base j at bits [2j, 2j+2); ~0 = empty (never canonical)
    uint32_t cls;        // bits 0-28 class id (or index into dual[] when kClsDual); kClsRc / kClsDual / kClsSpill
    uint32_t off;        // index into positions[]: first position in each member of the class
};
static_assert(sizeof(Entry) == 16, "entry must be half a sector");
constexpr uint32_t kClsSpill = 1u << 29;   // entry 0 of a bucket only: a key homed here lives in its second bucket
constexpr uint32_t kClsRc = 1u << 30;      // the library holds revcomp(key), not key itself
constexpr uint32_t kClsDual = 1u << 31;    // the library holds both strands: cls = index into dual[]
constexpr uint32_t kClsIdMask = kClsSpill - 1;
struct DualRec { uint32_t cls_s, off_s, cls_r, off_r; };   // key's own strand / its reverse complement

// Equivalence class = sparse bitset over references: sorted (word index, 32 member bits) pairs.
// One 32 B record (one sector) holds up to 4 pairs inline; wider classes point into ov_*.
struct ClassRec {
    uint32_t b[4];       // inline: member bits (unused = 0).  overflow: b[0] = offset into ov_w/ov_b/ov_pre, b[1] = pairs
    uint32_t w01, w23;   // inline: word indices, 16 bits each, ascending (unused = 0xFFFF, matches no word)
    uint32_t meta;       // bits 0-7: pairs (inline form); bit 31: overflow form
    uint32_t spare;
};
static_assert(sizeof(ClassRec) == 32, "class record must be one sector");
constexpr uint32_t kNoWord = 0xFFFFu;
constexpr uint32_t kRecOverflow = 1u << 31;
constexpr int kRecInline = 4;
constexpr uint64_t kEmptyKey = ~0ull;

struct HostLibrary {
    nb200_config cfg{};
    bool has_index = false;
    // --trim <TARGET_LENGTH>:<STRICTNESS> for this library (nb200_library_set_trim; file-level calls only)
    bool trim_on = false;
    int trim_target = 0;
    double trim_strictness = 0.0;
    // features
    std::vector<std::string> feature_names;   // ascending byte order; id = rank
    std::vector<uint32_t> tok_end, tok_comma; // rank of name+NUL / name+',' among all 2F tokens
    // references, INTERNAL order = (feature id, input order): ref -> feature is monotone
    std::vector<std::string> ref_names;
    std::vector<uint32_t> ref_feature;
    std::vector<uint32_t> ref_len, ref_gstart;
    bool identity_features = false;           // feature id == internal ref id
    // index images
    uint32_t n_refs = 0, n_features = 0, n_words = 1;
    uint64_t n_kmers = 0, n_classes = 0, n_buckets = 0, n_spilled = 0;
    std::vector<Entry> table;               // 2 * n_buckets
    std::vector<DualRec> dual;
    std::vector<ClassRec> class_rec;          // n_classes
    std::vector<uint32_t> ov_w, ov_b, ov_pre; // overflow pairs: word index, bits, members before the pair
    std::vector<uint32_t> positions;
    std::vector<uint64_t> ref2bit;            // global coordinate space, 32 bases / word
    std::vector<uint32_t> refN;               // 1 = not ACGT (or padding), 32 bases / word
    uint64_t total_gbases = 0;
};

// ---- device image: the index as one slab in HBM, and as the image section of an index file ----------------------
// Parts at 256-byte aligned offsets, hottest first (the L2 persistence window may only cover a prefix).  Any change to
// this layout, to Entry / ClassRec / DualRec or to hash_kmer / kmer_mix must bump kIndexVersion.
enum ImagePart { kPartTable, kPartClassRec, kPartOvW, kPartOvB, kPartOvPre, kPartPositions, kPartRefGstart, kPartRefFeature,
                 kPartRef2bit, kPartRefN, kPartDual, kImageParts };
struct ImageLayout {
    uint64_t bytes[kImageParts] = {};     // payload of each part
    uint64_t off[kImageParts] = {};
    uint64_t total = 0;                   // image size; a multiple of 256
};
ImageLayout image_layout(const uint64_t bytes[kImageParts]);
ImageLayout image_layout(const HostLibrary &L);      // of L's host images
// image bytes [offset, offset + len) of L's host images, padding as zeros
void image_fill(const HostLibrary &L, const ImageLayout &lay, uint64_t offset, uint64_t len, uint8_t *dst);
// L without its host images (what a device library keeps once its image is uploaded)
HostLibrary library_meta(const HostLibrary &L);

// ---- index file (.nb200idx, little-endian): header, host sections, the device image byte for byte --------------
constexpr uint32_t kIndexVersion = 1;
enum IndexSectionId { kSecFeatureNames, kSecTokEnd, kSecTokComma, kSecImage, kIndexSections };
struct IndexSection { uint64_t off, bytes, sum; };    // sum: index_checksum over the section's words
struct IndexHeader {
    char magic[8];                        // "NB200IDX"
    uint32_t version, header_bytes;
    uint32_t sizeof_entry, sizeof_classrec, sizeof_dualrec, k;
    int32_t score_threshold, score_filter, num_mismatches, discard_multiple_matches, intersect_level, discard_multi_hits,
        require_valid_pair, max_hits_to_report;   // the library JSON's config (strand_filter is a call parameter)
    double score_percent;
    uint32_t n_refs, n_features, n_words, identity_features;
    uint64_t n_kmers, n_classes, n_buckets, n_spilled, total_gbases;
    uint64_t json_bytes, json_fnv1a;      // the source JSON (provenance only)
    char lib_version[64];                 // nb200_version() of the writer
    uint64_t part_bytes[kImageParts];
    IndexSection sec[kIndexSections];
    uint64_t file_bytes;
    uint64_t header_sum;                  // index_checksum of the header with this field 0
};
static_assert(sizeof(IndexHeader) == 408, "index header has no padding");

// sum over the 64-bit words of p[0, bytes) (a partial last word is zero-padded), word i counted as word0 + i
uint64_t index_checksum(const void *p, uint64_t bytes, uint64_t word0, int threads = 1);
bool is_index_file(const std::string &path);
void write_index_file(const HostLibrary &L, const std::string &json_path, const std::string &out_path, int threads);
// An opened index file: header and host sections read and checked (a damaged or foreign file throws); the image is
// read on demand.
struct IndexFile {
    IndexHeader h{};
    int fd = -1;
    std::string path;
    IndexFile() = default;
    IndexFile(const IndexFile &) = delete;
    IndexFile &operator=(const IndexFile &) = delete;
    ~IndexFile();
    void read_image(uint64_t offset, uint64_t len, uint8_t *dst) const;
};
void open_index_file(const std::string &path, IndexFile &f, HostLibrary &meta);
// nb200_index_info with verify = 1: the image section's checksum, then every valid k-mer of every reference must look
// up (host_lookup) to a class that holds that reference.  Throws on a mismatch.
void verify_index_file(const IndexFile &f, const HostLibrary &meta, int threads);

uint64_t hash_kmer(uint64_t x);        // a change here or in kmer_mix (kmer_hash.hpp) must bump kIndexVersion
uint64_t revcomp_kmer(uint64_t x, int k);

// throws std::runtime_error (EINVAL-class) / LimitError
struct LimitError : std::runtime_error { using std::runtime_error::runtime_error; };

void parse_library_json(const std::string &path, std::vector<std::string> &names, std::vector<std::string> &seqs,
                        std::vector<std::string> &features, nb200_config &cfg);
void build_library(const std::vector<std::string> &names, const std::vector<std::string> &seqs,
                   const std::vector<std::string> &features, const nb200_config &cfg, int host_threads,
                   HostLibrary &out, bool verify = false);
void host_lookup(const HostLibrary &L, uint64_t x, uint32_t cl[2], uint32_t of[2]);
void build_feature_dictionary(const std::vector<std::string> &sorted_names, HostLibrary &out);
int parse_strand_filter(const char *s);

}  // namespace nb200
