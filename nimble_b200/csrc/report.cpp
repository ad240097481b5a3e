// Host side of `nimble report` (nimble/__main__.py:213-293): per-read TSV -> rows for the device
// UMI stage (agg.cuh) -> counts TSV.  The arithmetic (merge, thresholding, intersection, counting)
// runs on the GPU; this file only parses, interns strings and writes.
#include "ingest.hpp"
#include "library.hpp"
#include "pandas_na.hpp"
#include "umi_code.hpp"

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <string_view>
#include <unordered_map>

namespace nb200 {

void slurp_maybe_gz(const std::string &path, std::string &out);   // ingest.cpp

// strings -> dense ids in ascending byte order (pandas groupby order == output order of the counts TSV)
static void intern_sorted(const std::vector<std::string_view> &vals, std::vector<uint32_t> &ids, std::vector<std::string> &uniq) {
    std::unordered_map<std::string_view, uint32_t> seen;
    seen.reserve(vals.size() / 4 + 16);
    std::vector<std::string_view> keys;
    for (auto v : vals) if (seen.emplace(v, 0u).second) keys.push_back(v);
    std::sort(keys.begin(), keys.end());
    uniq.clear();
    uniq.reserve(keys.size());
    for (uint32_t i = 0; i < keys.size(); i++) { seen[keys[i]] = i; uniq.emplace_back(keys[i]); }
    ids.resize(vals.size());
    for (size_t i = 0; i < vals.size(); i++) ids[i] = seen[vals[i]];
}

// strings -> dense ids in ascending byte order with few distinct values (cells, feature names): per-thread distinct sets,
// one merged sorted dictionary, ids looked up in parallel
static void intern_sorted_mt(const std::vector<std::string_view> &vals, std::vector<uint32_t> &ids, std::vector<std::string> &uniq, int T) {
    const size_t n = vals.size();
    if (T <= 1 || n < 200000) { intern_sorted(vals, ids, uniq); return; }
    std::vector<std::vector<std::string_view>> local((size_t)T);
    parallel_for(T, [&](int t) {
        const size_t a = n * (size_t)t / T, b = n * (size_t)(t + 1) / T;
        std::unordered_map<std::string_view, uint32_t> seen;
        for (size_t i = a; i < b; i++) if (seen.emplace(vals[i], 0u).second) local[(size_t)t].push_back(vals[i]);
    });
    std::vector<std::string_view> keys;
    for (auto &l : local) keys.insert(keys.end(), l.begin(), l.end());
    std::sort(keys.begin(), keys.end());
    keys.erase(std::unique(keys.begin(), keys.end()), keys.end());
    std::unordered_map<std::string_view, uint32_t> dict;
    dict.reserve(keys.size() * 2 + 16);
    uniq.clear();
    uniq.reserve(keys.size());
    for (uint32_t i = 0; i < keys.size(); i++) { dict.emplace(keys[i], i); uniq.emplace_back(keys[i]); }
    ids.resize(n);
    parallel_for(T, [&](int t) {
        const size_t a = n * (size_t)t / T, b = n * (size_t)(t + 1) / T;
        for (size_t i = a; i < b; i++) ids[i] = dict.find(vals[i])->second;
    });
}

// UMI strings -> ids (umi_code.hpp): an ACGTN UMI of 1..13 bases is its code, any other is interned with bit 31 set.
// Only equality matters (the UMI order never reaches the output).
static void umi_ids(const std::vector<std::string_view> &vals, std::vector<uint32_t> &ids, int T) {
    const size_t n = vals.size();
    ids.resize(n);
    const int P = n < 100000 ? 1 : std::max(1, T);
    parallel_for(P, [&](int t) {
        const size_t a = n * (size_t)t / P, b = n * (size_t)(t + 1) / P;
        for (size_t i = a; i < b; i++) if (!umi_code(vals[i], ids[i])) ids[i] = 0;       // 0: no code (codes start at 1)
    });
    std::vector<std::string_view> other;
    std::vector<size_t> at;
    for (size_t i = 0; i < n; i++) if (!ids[i]) { other.push_back(vals[i]); at.push_back(i); }
    if (other.empty()) return;
    std::vector<uint32_t> oid;
    std::vector<std::string> names;
    intern_sorted(other, oid, names);
    if (names.size() >= kUmiInterned) throw LimitError("more than 2^31 distinct UMIs that are not ACGTN of up to 13 bases");
    for (size_t j = 0; j < at.size(); j++) ids[at[j]] = oid[j] | kUmiInterned;
}

std::vector<size_t> line_pieces(const std::string &t, size_t body, int threads) {
    const int T = (t.size() - body < (4u << 20)) ? 1 : std::max(1, threads);
    std::vector<size_t> cut((size_t)T + 1, t.size());
    cut[0] = body;
    for (int k = 1; k < T; k++) {
        size_t p = body + (t.size() - body) * (size_t)k / T;
        p = std::max(p, cut[(size_t)k - 1]);
        const size_t e = t.find('\n', p);
        cut[(size_t)k] = e == std::string::npos ? t.size() : e + 1;
    }
    return cut;
}

// returns false when there is nothing to report (empty file / header only / no usable row)
bool parse_per_read_tsv(const std::string &path, ReportRows &R, int threads) {
    slurp_maybe_gz(path, R.text);
    const std::string &t = R.text;
    if (t.empty()) return false;
    auto split = [](std::string_view line, std::vector<std::string_view> &out) {
        out.clear();
        size_t a = 0;
        for (;;) {
            const size_t e = line.find('\t', a);
            if (e == std::string_view::npos) { out.push_back(line.substr(a)); break; }
            out.push_back(line.substr(a, e - a));
            a = e + 1;
        }
    };
    // header
    size_t hdr_end = t.find('\n');
    if (hdr_end == std::string::npos) hdr_end = t.size();
    std::vector<std::string_view> f;
    {
        size_t b = hdr_end;
        if (b > 0 && t[b - 1] == '\r') b--;
        split(std::string_view(t.data(), b), f);
    }
    int fi = -1, ui = -1, ci = -1, si = -1;
    for (int i = 0; i < (int)f.size(); i++) {
        if (f[i] == "nimble_features") fi = i; else if (f[i] == "r1_UB") ui = i;
        else if (f[i] == "r1_CB") ci = i; else if (f[i] == "nimble_score") si = i;
    }
    if (fi < 0 || ui < 0 || ci < 0 || si < 0) throw std::runtime_error("per-read TSV lacks nimble_features / r1_UB / r1_CB / nimble_score");
    const int need = std::max(std::max(fi, ui), std::max(ci, si));
    const size_t body = std::min(t.size(), hdr_end + 1);
    // every thread parses the lines of its piece into its own vectors
    const std::vector<size_t> cut = line_pieces(t, body, threads);
    const int T = (int)cut.size() - 1;
    struct Part { std::vector<std::string_view> cb, umi, feat; std::vector<double> score; };
    std::vector<Part> parts((size_t)T);
    parallel_for(T, [&](int k) {
        Part &P = parts[(size_t)k];
        std::vector<std::string_view> g;
        size_t p = cut[(size_t)k];
        const size_t end = cut[(size_t)k + 1];
        std::string num;
        while (p < end) {
            const void *nl = memchr(t.data() + p, '\n', end - p);
            const size_t e = nl ? (size_t)((const char *)nl - t.data()) : end;
            size_t b = e;
            if (b > p && t[b - 1] == '\r') b--;
            const std::string_view line(t.data() + p, b - p);
            p = e + 1;
            split(line, g);
            if ((int)g.size() <= need) continue;                 // short row: its missing cells are NaN (dropna, :244)
            if (pandas_na(g[fi]) || pandas_na(g[ui]) || pandas_na(g[ci]) || pandas_na(g[si])) continue;
            double sc;
            if (g[si].size() == 1 && g[si][0] >= '0' && g[si][0] <= '9') sc = (double)(g[si][0] - '0');   // the aligner writes "1"
            else {
                num.assign(g[si]);
                char *endp = nullptr;
                sc = strtod(num.c_str(), &endp);
                if (endp == num.c_str() || *endp != '\0' || sc != sc) continue;
            }
            P.cb.push_back(g[ci]); P.umi.push_back(g[ui]); P.feat.push_back(g[fi]);
            P.score.push_back(sc);
        }
    });
    std::vector<size_t> base((size_t)T + 1, 0);
    for (int k = 0; k < T; k++) base[(size_t)k + 1] = base[(size_t)k] + parts[(size_t)k].cb.size();
    const size_t n = base[(size_t)T];
    if (!n) return false;
    if (n > 0xFFFFFFF0ull) throw std::runtime_error("more than 2^32 rows in the per-read TSV");
    std::vector<std::string_view> cbs(n), umis(n), feats(n);
    R.score.resize(n);
    parallel_for(T, [&](int k) {
        const Part &P = parts[(size_t)k];
        const size_t o = base[(size_t)k];
        std::copy(P.cb.begin(), P.cb.end(), cbs.begin() + o);
        std::copy(P.umi.begin(), P.umi.end(), umis.begin() + o);
        std::copy(P.feat.begin(), P.feat.end(), feats.begin() + o);
        std::copy(P.score.begin(), P.score.end(), R.score.begin() + o);
    });
    parts.clear();
    // feature names: every comma-separated token of every row
    std::vector<uint32_t> row_off(n + 1, 0);
    const int T2 = n < 100000 ? 1 : std::max(1, threads);
    std::vector<uint64_t> tok_base((size_t)T2 + 1, 0);
    parallel_for(T2, [&](int k) {                                // tokens per row
        const size_t a = n * (size_t)k / T2, b = n * (size_t)(k + 1) / T2;
        uint64_t tot = 0;
        for (size_t i = a; i < b; i++) {
            uint32_t cnt = 1;
            for (char ch : feats[i]) cnt += ch == ',';
            row_off[i + 1] = cnt;
            tot += cnt;
        }
        tok_base[(size_t)k + 1] = tot;
    });
    for (int k = 0; k < T2; k++) tok_base[(size_t)k + 1] += tok_base[(size_t)k];
    if (tok_base[(size_t)T2] > 0xFFFFFFF0ull) throw std::runtime_error("more than 2^32 feature names in the per-read TSV");
    std::vector<std::string_view> toks((size_t)tok_base[(size_t)T2]);
    parallel_for(T2, [&](int k) {
        const size_t a = n * (size_t)k / T2, b = n * (size_t)(k + 1) / T2;
        uint64_t at = tok_base[(size_t)k];
        for (size_t i = a; i < b; i++) {
            const uint32_t cnt = row_off[i + 1];
            row_off[i + 1] = (uint32_t)(at + cnt);               // exclusive end of row i
            std::string_view v = feats[i];
            size_t p0 = 0;
            for (;;) {
                const size_t e = v.find(',', p0);
                toks[(size_t)at++] = v.substr(p0, e == std::string_view::npos ? std::string_view::npos : e - p0);
                if (e == std::string_view::npos) break;
                p0 = e + 1;
            }
        }
    });
    std::vector<uint32_t> tok_ids;
    intern_sorted_mt(toks, tok_ids, R.feature_names, threads);
    parallel_for(T2, [&](int k) {                                // sorted names inside a row (:248)
        const size_t a = n * (size_t)k / T2, b = n * (size_t)(k + 1) / T2;
        for (size_t i = a; i < b; i++) if (row_off[i + 1] - row_off[i] > 1) std::sort(tok_ids.begin() + row_off[i], tok_ids.begin() + row_off[i + 1]);
    });
    R.off = std::move(row_off);
    R.ids = std::move(tok_ids);
    std::vector<uint32_t> cid, uid;
    intern_sorted_mt(cbs, cid, R.cells, threads);
    umi_ids(umis, uid, threads);
    R.key.resize(n);
    parallel_for(T2, [&](int k) {
        const size_t a = n * (size_t)k / T2, b = n * (size_t)(k + 1) / T2;
        for (size_t i = a; i < b; i++) R.key[i] = ((uint64_t)cid[i] << 32) | uid[i];
    });
    return true;
}

void write_counts_tsv(const std::string &out_path, const nb200_counts *c, const std::vector<std::string> &feature_names,
                      const std::vector<std::string> &cells) {
    const std::string tmp = out_path + ".tmp";
    FILE *f = fopen(tmp.c_str(), "wb");
    if (!f) throw IoError("cannot write " + tmp);
    std::string buf;
    const uint64_t n = c ? c->n_rows : 0;
    for (uint64_t i = 0; i < n; i++) {
        for (uint32_t j = c->feat_off[i]; j < c->feat_off[i + 1]; j++) { if (j > c->feat_off[i]) buf += ','; buf += feature_names[c->feat_ids[j]]; }
        buf += '\t'; buf += std::to_string(c->count[i]); buf += '\t'; buf += cells[c->cell[i]]; buf += '\n';
        if (buf.size() > (1u << 22)) { if (fwrite(buf.data(), 1, buf.size(), f) != buf.size()) { fclose(f); throw IoError("write failed on " + tmp); } buf.clear(); }
    }
    if (!buf.empty() && fwrite(buf.data(), 1, buf.size(), f) != buf.size()) { fclose(f); throw IoError("write failed on " + tmp); }
    if (fclose(f) != 0) throw IoError("close failed on " + tmp);
    if (rename(tmp.c_str(), out_path.c_str()) != 0) throw IoError("cannot rename " + tmp);
}

}  // namespace nb200
