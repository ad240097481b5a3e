// Host side of `nimble fastq-to-bam` (SURVEY.md §8a A5): paired 10x FASTQ(.gz) with qualities in,
// process_pair's skip rules (nimble/fastq_barcode_processor.py:152-165), unaligned BAM with CB/UB
// tags out (:186-207, header :235-238).  The barcode correction itself runs on the GPU
// (barcode.cuh); this file only parses, slices and serialises.  BGZF is written block-parallel
// with zlib, no htslib.
#include "ingest.hpp"

#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <cctype>
#include <cstdio>
#include <cstring>
#include <thread>

namespace nb200 {

void slurp_maybe_gz(const std::string &path, std::string &out);   // ingest.cpp

// 4-line FASTQ records (what 10x pipelines emit); record.id = title up to the first whitespace
void load_fastq_qual(const std::string &path, FastqQ &F) {
    slurp_maybe_gz(path, F.text);
    const char *base = F.text.data(), *p = base, *end = base + F.text.size();
    while (p < end) {
        if (*p == '\n' || *p == '\r') { p++; continue; }             // blank lines between records
        if (*p != '@') throw IoError("malformed FASTQ record in " + path);
        const char *l[4], *e[4];
        bool more = true;                                            // another line starts at p
        for (int k = 0; k < 4; k++) {
            if (!more) {
                if (k < 3) throw IoError("truncated FASTQ record in " + path);
                l[k] = e[k] = end;                                   // empty quality line at end of file
                continue;
            }
            l[k] = p;
            const char *nl = p < end ? (const char *)memchr(p, '\n', end - p) : nullptr;
            e[k] = nl ? nl : end;
            more = nl != nullptr;
            p = nl ? nl + 1 : end;
            while (e[k] > l[k] && e[k][-1] == '\r') e[k]--;
        }
        if (l[2] >= end || *l[2] != '+') throw IoError("malformed FASTQ record (no '+' line) in " + path);
        const char *ne = l[0] + 1;
        while (ne < e[0] && *ne != ' ' && *ne != '\t') ne++;
        if ((e[3] - l[3]) != (e[1] - l[1])) throw IoError("FASTQ sequence and quality lengths differ in " + path);
        FqRec r;
        r.name = (uint64_t)(l[0] + 1 - base); r.name_len = (uint32_t)(ne - (l[0] + 1));
        r.seq = (uint64_t)(l[1] - base); r.len = (uint32_t)(e[1] - l[1]);
        r.qual = (uint64_t)(l[3] - base);
        F.recs.push_back(r);
    }
}

// process_pair up to the correction call: eligibility + the three skip counters; cb/qual are n x cb_len
// (zero-filled for ineligible pairs), qual holds phred values (ASCII - 33)
void slice_barcodes(const FastqQ &A, const FastqQ &B, int cb_len, int umi_len, int threads, uint8_t *cb, uint8_t *qual,
                    uint8_t *eligible, nb200_cb_stats &st) {
    const size_t n = std::min(A.recs.size(), B.recs.size());          // zip() stops at the shorter file
    std::atomic<uint64_t> mism{0}, tshort{0}, norem{0};
    auto work = [&](size_t a, size_t b) {
        uint64_t m = 0, t = 0, r = 0;
        for (size_t i = a; i < b; i++) {
            const FqRec &x = A.recs[i], &y = B.recs[i];
            uint8_t *c = cb + i * (size_t)cb_len, *q = qual + i * (size_t)cb_len;
            eligible[i] = 0;
            memset(c, 0, (size_t)cb_len); memset(q, 0, (size_t)cb_len);
            if (!name_eq_stripped(A.text.data() + x.name, x.name_len, B.text.data() + y.name, y.name_len)) { m++; continue; }
            if (x.len < (uint32_t)(cb_len + umi_len)) { t++; continue; }
            if (x.len == (uint32_t)(cb_len + umi_len)) { r++; continue; }
            eligible[i] = 1;
            memcpy(c, A.text.data() + x.seq, (size_t)cb_len);
            const char *qs = A.text.data() + x.qual;
            for (int j = 0; j < cb_len; j++) q[j] = (uint8_t)(qs[j] - 33);
        }
        mism += m; tshort += t; norem += r;
    };
    const int T = std::max(1, threads);
    if (T == 1 || n < 65536) work(0, n);
    else {
        std::vector<std::thread> th;
        const size_t per = (n + T - 1) / T;
        for (int t = 0; t < T; t++) th.emplace_back(work, std::min(n, t * per), std::min(n, (t + 1) * per));
        for (auto &x : th) x.join();
    }
    st.total_pairs = n; st.name_mismatch = mism; st.too_short = tshort; st.no_remaining_seq = norem;
}

// ---- BAM / BGZF writer ----------------------------------------------------------------------------
static void put32(std::string &s, uint32_t v) { char b[4] = {(char)v, (char)(v >> 8), (char)(v >> 16), (char)(v >> 24)}; s.append(b, 4); }
static void put16(std::string &s, uint32_t v) { char b[2] = {(char)v, (char)(v >> 8)}; s.append(b, 2); }

static const uint8_t *nt16_table() {      // built once, thread-safe (C++11 magic static): the BAM writer's workers all call it
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

static void bam_record(std::string &out, const char *name, uint32_t name_len, uint32_t flag, const char *seq, const char *qual,
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

static void bgzf_blocks(const std::string &raw, std::string &out) {
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

void write_10x_bam(const std::string &out_path, const FastqQ &A, const FastqQ &B, int cb_len, int umi_len, const int32_t *idx,
                   const uint8_t *status, const std::vector<std::string> &wl_entries, int threads, nb200_cb_stats &st) {
    const size_t n = std::min(A.recs.size(), B.recs.size());
    const std::string tmp = out_path + ".tmp";
    FILE *f = fopen(tmp.c_str(), "wb");
    if (!f) throw IoError("cannot write " + tmp);
    auto emit = [&](const std::string &s) {
        if (!s.empty() && fwrite(s.data(), 1, s.size(), f) != s.size()) { fclose(f); throw IoError("write error on " + tmp); }
    };
    {   // header :235-238, as pysam serialises the dict
        const std::string text = "@HD\tVN:1.6\tSO:queryname\n@PG\tID:nimble-fastq-to-bam\tPN:nimble\tVN:1.2\tCL:whitelist-based CB correction\n";
        std::string raw("BAM\1", 4), z;
        put32(raw, (uint32_t)text.size()); raw += text; put32(raw, 0);
        bgzf_blocks(raw, z);
        emit(z);
    }
    const size_t kChunk = 1 << 15;                                   // pairs per work item
    const size_t n_chunks = (n + kChunk - 1) / kChunk;
    const int T = (int)std::max<size_t>(1, std::min<size_t>((size_t)std::max(1, threads), n_chunks));
    std::atomic<uint64_t> written{0};
    for (size_t c0 = 0; c0 < n_chunks; c0 += (size_t)T) {            // T chunks compressed in parallel, written in order
        const size_t nc = std::min((size_t)T, n_chunks - c0);
        std::vector<std::string> z(nc);
        std::vector<std::string> errs(nc);
        auto work = [&](size_t k) {
            try {
                std::string raw;
                uint64_t w = 0;
                const size_t a = (c0 + k) * kChunk, b = std::min(n, a + kChunk);
                for (size_t i = a; i < b; i++) {
                    if (status[i] != NB200_CB_PERFECT && status[i] != NB200_CB_CORRECTED) continue;
                    const FqRec &x = A.recs[i], &y = B.recs[i];
                    const char *t1 = A.text.data(), *t2 = B.text.data();
                    uint32_t nl = x.name_len;
                    if (nl >= 2 && t1[x.name + nl - 2] == '/' && t1[x.name + nl - 1] == '1') nl -= 2;
                    if (nl > 254) throw IoError("read name longer than 254 bytes");
                    const std::string &cbs = wl_entries[(size_t)idx[i]];
                    const uint32_t bl = (uint32_t)(cb_len + umi_len);
                    bam_record(raw, t1 + x.name, nl, 77, t1 + x.seq + bl, t1 + x.qual + bl, x.len - bl, cbs.data(),
                               (uint32_t)cbs.size(), t1 + x.seq + cb_len, (uint32_t)umi_len);
                    bam_record(raw, t1 + x.name, nl, 141, t2 + y.seq, t2 + y.qual, y.len, cbs.data(), (uint32_t)cbs.size(),
                               t1 + x.seq + cb_len, (uint32_t)umi_len);
                    w++;
                }
                bgzf_blocks(raw, z[k]);
                written += w;
            } catch (const std::exception &e) { errs[k] = e.what(); }
        };
        std::vector<std::thread> th;
        for (size_t k = 0; k < nc; k++) th.emplace_back(work, k);
        for (auto &x : th) x.join();
        for (size_t k = 0; k < nc; k++) {
            if (!errs[k].empty()) { fclose(f); remove(tmp.c_str()); throw IoError(errs[k]); }
            emit(z[k]);
        }
    }
    static const unsigned char eof[28] = {0x1f, 0x8b, 0x08, 0x04, 0, 0, 0, 0, 0, 0xff, 0x06, 0, 0x42, 0x43, 0x02, 0,
                                          0x1b, 0, 0x03, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    emit(std::string((const char *)eof, 28));
    if (fclose(f) != 0) throw IoError("close failed on " + tmp);
    if (rename(tmp.c_str(), out_path.c_str()) != 0) throw IoError("cannot rename " + tmp);
    st.written_pairs = written;
}

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
