// What `nimble fastq-to-bam` (SURVEY.md §8a A5) writes: unaligned BAM records with CB/UB tags (:186-207, header
// :235-238) in BGZF blocks (zlib, no htslib), and its whitelist reader.  The streaming pipeline (stream.cpp, 10x mode)
// applies process_pair's rules, corrects the barcodes on the GPU (barcode.cuh) and calls these from its format tasks.
#include "ingest.hpp"

#include <zlib.h>

#include <algorithm>
#include <cctype>
#include <cstring>

namespace nb200 {

void slurp_maybe_gz(const std::string &path, std::string &out);   // ingest.cpp

// ---- BAM / BGZF writer ----------------------------------------------------------------------------
static void put32(std::string &s, uint32_t v) { char b[4] = {(char)v, (char)(v >> 8), (char)(v >> 16), (char)(v >> 24)}; s.append(b, 4); }
static void put16(std::string &s, uint32_t v) { char b[2] = {(char)v, (char)(v >> 8)}; s.append(b, 2); }

static const uint8_t *nt16_table() {      // built once, thread-safe (C++11 magic static): the format tasks all call it
    struct Table {
        uint8_t t[256];
        Table() {
            memset(t, 15, sizeof t);
            const char *codes = "=ACMGRSVTWYHKDBN";
            for (int i = 0; i < 16; i++) { t[(uint8_t)codes[i]] = (uint8_t)i; t[(uint8_t)tolower(codes[i])] = (uint8_t)i; }
        }
    };
    static const Table table;
    return table.t;
}

void bam_record(std::string &out, const char *name, uint32_t name_len, uint32_t flag, const char *seq, const char *qual,
                       uint32_t len, const char *cb, uint32_t cb_len, const char *ub, uint32_t ub_len) {
    const uint8_t *nt = nt16_table();
    const uint32_t l_name = name_len + 1;
    const uint32_t body = 32 + l_name + (len + 1) / 2 + len + (3 + cb_len + 1) + (3 + ub_len + 1);
    put32(out, body);
    put32(out, (uint32_t)-1);            // refID
    put32(out, (uint32_t)-1);            // pos
    out.push_back((char)l_name);         // l_read_name
    out.push_back(0);                    // mapq
    put16(out, 4680);                    // bin of an unplaced read
    put16(out, 0);                       // n_cigar_op
    put16(out, flag);
    put32(out, len);
    put32(out, (uint32_t)-1);            // next refID
    put32(out, (uint32_t)-1);            // next pos
    put32(out, 0);                       // tlen
    out.append(name, name_len); out.push_back('\0');
    for (uint32_t i = 0; i < len; i += 2) {
        const uint8_t hi = nt[(uint8_t)seq[i]], lo = i + 1 < len ? nt[(uint8_t)seq[i + 1]] : 0;
        out.push_back((char)((hi << 4) | lo));
    }
    for (uint32_t i = 0; i < len; i++) out.push_back((char)(qual[i] - 33));
    out.append("CBZ", 3); out.append(cb, cb_len); out.push_back('\0');
    out.append("UBZ", 3); out.append(ub, ub_len); out.push_back('\0');
}

void bgzf_blocks(const std::string &raw, std::string &out) {
    const size_t kMax = 0xff00;
    for (size_t p = 0; p < raw.size(); p += kMax) {
        const size_t n = std::min(kMax, raw.size() - p);
        unsigned char buf[65536 + 1024];
        z_stream zs;
        memset(&zs, 0, sizeof zs);
        if (deflateInit2(&zs, 6, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY) != Z_OK) throw IoError("deflateInit2 failed");
        zs.next_in = (Bytef *)raw.data() + p; zs.avail_in = (uInt)n;
        zs.next_out = buf; zs.avail_out = sizeof buf;
        const int rc = deflate(&zs, Z_FINISH);
        const size_t clen = zs.total_out;
        deflateEnd(&zs);
        if (rc != Z_STREAM_END || clen + 26 > 65536) throw IoError("BGZF block does not fit");
        const unsigned char hdr[16] = {31, 139, 8, 4, 0, 0, 0, 0, 0, 255, 6, 0, 'B', 'C', 2, 0};
        out.append((const char *)hdr, 16);
        put16(out, (uint32_t)(clen + 25));
        out.append((const char *)buf, clen);
        put32(out, (uint32_t)crc32(crc32(0L, Z_NULL, 0), (const Bytef *)raw.data() + p, (uInt)n));
        put32(out, (uint32_t)n);
    }
}

std::string bam_header_bgzf() {   // :235-238, as pysam serialises the dict
    const std::string text = "@HD\tVN:1.6\tSO:queryname\n@PG\tID:nimble-fastq-to-bam\tPN:nimble\tVN:1.2\tCL:whitelist-based CB correction\n";
    std::string raw("BAM\1", 4), z;
    put32(raw, (uint32_t)text.size()); raw += text; put32(raw, 0);
    bgzf_blocks(raw, z);
    return z;
}

const unsigned char kBgzfEof[28] = {0x1f, 0x8b, 0x08, 0x04, 0, 0, 0, 0, 0, 0xff, 0x06, 0, 0x42, 0x43, 0x02, 0,
                                    0x1b, 0, 0x03, 0, 0, 0, 0, 0, 0, 0, 0, 0};

// load_cb_whitelist (:38-71): stripped non-empty lines
void read_whitelist_lines(const std::string &path, std::vector<std::string> &lines) {
    std::string text;
    slurp_maybe_gz(path, text);
    size_t p = 0;
    while (p < text.size()) {
        size_t e = text.find('\n', p);
        if (e == std::string::npos) e = text.size();
        size_t a = p, b = e;
        auto ws = [](char c) { return c == ' ' || c == '\t' || c == '\r' || c == '\n' || c == '\v' || c == '\f'; };
        while (a < b && ws(text[a])) a++;
        while (b > a && ws(text[b - 1])) b--;
        if (b > a) lines.emplace_back(text, a, b - a);
        p = e + 1;
    }
}

}  // namespace nb200
