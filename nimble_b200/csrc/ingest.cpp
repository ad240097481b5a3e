// Whole-file reads (slurp_maybe_gz: the whitelist, report, report -s).  The aligner's file entries, fastq-to-bam and
// `align --map` stream their input instead (stream.cpp).
#include "ingest.hpp"

#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstring>
#include <thread>

namespace nb200 {

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

}  // namespace nb200
