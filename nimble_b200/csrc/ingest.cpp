// Whole-file reads (slurp_maybe_gz: fastq-to-bam, the 10x one-pass route, report) and the per-read TSV of the 10x one-pass
// route (nb200_align_10x_fastq, `align --map`).  The aligner's file entries stream their input instead (stream.cpp).
#include "ingest.hpp"

#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstring>
#include <thread>

namespace nb200 {

static bool ends_with(const std::string &s, const char *suf) {
    const size_t n = strlen(suf);
    return s.size() >= n && s.compare(s.size() - n, n, suf) == 0;
}

// whole (optionally gzip-compressed) file -> memory; gzread handles plain files transparently
static void slurp_gz(const std::string &path, std::string &out) {
    gzFile f = gzopen(path.c_str(), "rb");
    if (!f) throw IoError("cannot open " + path);
    gzbuffer(f, 1 << 20);
    out.clear();
    std::vector<char> buf(1 << 22);
    for (;;) {
        int n = gzread(f, buf.data(), (unsigned)buf.size());
        if (n < 0) { gzclose(f); throw IoError("read error in " + path); }
        if (n == 0) break;
        out.append(buf.data(), (size_t)n);
    }
    gzclose(f);
}

// plain files (the per-read TSV of `align` is hundreds of MB): sized once, read in slices by a few threads straight into
// place (gzread would copy every byte twice more and the string would be regrown a dozen times); gzip input: slurp_gz
void slurp_maybe_gz(const std::string &path, std::string &out) {
    FILE *f = fopen(path.c_str(), "rb");
    if (!f) throw IoError("cannot open " + path);
    unsigned char magic[2] = {0, 0};
    const size_t got = fread(magic, 1, 2, f);
    const bool gz = got == 2 && magic[0] == 0x1f && magic[1] == 0x8b;
    long long size = -1;
    if (!gz && fseeko(f, 0, SEEK_END) == 0) size = (long long)ftello(f);
    fclose(f);
    if (gz || size < 0) { slurp_gz(path, out); return; }
    out.clear();
    out.resize((size_t)size);
    if (!size) return;
    const int T = (int)std::max<long long>(1, std::min<long long>(8, size / (32 << 20)));
    std::vector<std::thread> th;
    std::atomic<int> bad{0};
    for (int t = 0; t < T; t++)
        th.emplace_back([&, t] {
            FILE *g = fopen(path.c_str(), "rb");
            if (!g) { bad = 1; return; }
            const size_t a = (size_t)size * (size_t)t / (size_t)T, b = (size_t)size * (size_t)(t + 1) / (size_t)T;
            if (fseeko(g, (off_t)a, SEEK_SET) != 0 || fread(&out[a], 1, b - a, g) != b - a) bad = 1;
            fclose(g);
        });
    for (auto &x : th) x.join();
    if (bad) throw IoError("read error in " + path);
}

void Arena::add(const char *p, size_t n) {
    data.append(p, n);
    off.push_back((int64_t)data.size());
}

// ---- TSV output ------------------------------------------------------------------------------------
struct Sink {
    FILE *f = nullptr;
    gzFile g = nullptr;
    std::string buf;
    void open(const std::string &path, bool gz) {
        if (gz) { g = gzopen(path.c_str(), "wb"); if (!g) throw IoError("cannot write " + path); gzbuffer(g, 1 << 20); }
        else { f = fopen(path.c_str(), "wb"); if (!f) throw IoError("cannot write " + path); }
    }
    void flush() {
        if (buf.empty()) return;
        if (g) { if (gzwrite(g, buf.data(), (unsigned)buf.size()) <= 0) throw IoError("write failed"); }
        else if (fwrite(buf.data(), 1, buf.size(), f) != buf.size()) throw IoError("write failed");
        buf.clear();
    }
    void put(const std::string &s) { buf += s; if (buf.size() > (1 << 22)) flush(); }
    void close() { flush(); if (g) gzclose(g); if (f) fclose(f); g = nullptr; f = nullptr; }
    ~Sink() { if (g) gzclose(g); if (f) fclose(f); }
};

void write_per_read_tsv(const std::string &out_path, const ReadSet &R, const nb200_read_result *res, const int32_t *feats,
                        int max_hits, const std::vector<std::string> &feature_names, int threads) {
    const std::string tmp = out_path + ".tmp";
    Sink s;
    s.open(tmp, ends_with(out_path, ".gz"));
    s.put("nimble_features\tnimble_score\tr1_forward_score\tr1_reverse_score\tr2_forward_score\tr2_reverse_score\t"
          "r1_QNAME\tr1_CB\tr1_UB\tr1_UR\tr1_GN\tr1_POS\tr2_POS\n");
    const size_t n = R.r1.size();
    // rows are formatted by all host threads in slabs and written in order
    const size_t kSlab = 1 << 16;
    const int T = std::max(1, threads);
    auto format = [&](size_t a, size_t b, std::string &out) {
        char num[24];
        for (size_t i = a; i < b; i++) {
            if (!res[i].n_feat) continue;
            for (int j = 0; j < res[i].n_feat; j++) { if (j) out += ','; out += feature_names[feats[i * (size_t)max_hits + j]]; }
            out += "\t1";
            for (int o = 0; o < 4; o++) { out += '\t'; out.append(num, (size_t)snprintf(num, sizeof num, "%u", (unsigned)res[i].score[o])); }
            out += '\t'; out.append(R.names.ptr(i), R.names.len(i));
            out += '\t'; out.append(R.cb.ptr(i), R.cb.len(i));
            out += '\t'; out.append(R.ub.ptr(i), R.ub.len(i));
            out += "\t\t\t\t\n";                           // r1_UR, r1_GN, r1_POS, r2_POS: unaligned records carry none
        }
    };
    for (size_t base = 0; base < n; base += kSlab * (size_t)T) {
        const size_t slabs = std::min<size_t>((size_t)T, (n - base + kSlab - 1) / kSlab);
        std::vector<std::string> outs(slabs);
        std::vector<std::thread> th;
        for (size_t k = 0; k < slabs; k++)
            th.emplace_back([&, k] { format(base + k * kSlab, std::min(n, base + (k + 1) * kSlab), outs[k]); });
        for (auto &x : th) x.join();
        for (auto &o : outs) s.put(o);
    }
    s.close();
    if (rename(tmp.c_str(), out_path.c_str()) != 0) throw IoError("cannot rename " + tmp);
}

}  // namespace nb200
