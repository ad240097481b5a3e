// Host side of `report -s` (summarize_fields, nimble/__main__.py:291-297): per-read TSV -> one typed key per cell for the
// device grouping (summarize.cuh) -> summary TSV, byte-identical to frontend.summarize_fields_tsv.  Reading, typing,
// equality and printing follow the Python path (DESIGN.md §2.13); grouping, counting and ordering run on the GPU.
#include "ingest.hpp"
#include "library.hpp"
#include "pandas_na.hpp"

#include <algorithm>
#include <charconv>
#include <cmath>
#include <cstring>
#include <string_view>
#include <unordered_map>

namespace nb200 {

void slurp_maybe_gz(const std::string &path, std::string &out);   // ingest.cpp

static inline std::string_view cell_view(const std::string &t, uint64_t c) { return std::string_view(t.data() + (c >> 24), c & 0xFFFFFF); }

// what Python's int() and float() strip from ASCII text: space and \t \n \v \f \r, not \x1c-\x1f (which str.strip() takes);
// bytes >= 0x80 make a cell a string (DESIGN.md §7)
static inline bool py_space(unsigned char ch) { return ch == ' ' || (ch >= '\t' && ch <= '\r'); }

static inline bool ascii_plain(std::string_view v) {           // no byte >= 0x80 and no '_'
    for (unsigned char ch : v) if (ch >= 0x80 || ch == '_') return false;
    return true;
}

static bool strict_int(std::string_view v) {                    // ASCII [+-]?[0-9]+
    size_t i = (!v.empty() && (v[0] == '+' || v[0] == '-')) ? 1 : 0;
    if (i == v.size()) return false;
    for (; i < v.size(); i++) if (v[i] < '0' || v[i] > '9') return false;
    return true;
}

struct IntText { bool neg; std::string_view digits; };          // canonical int: no sign for 0, no leading zeros ("" = 0)
static IntText canon_int(std::string_view v) {
    bool neg = v[0] == '-';
    size_t i = (v[0] == '+' || v[0] == '-') ? 1 : 0;
    while (i < v.size() && v[i] == '0') i++;
    std::string_view d = v.substr(i);
    if (d.empty()) neg = false;
    return {neg, d};
}

static double parse_decimal(std::string_view s) {               // [0-9]*[.[0-9]*][e[+-][0-9]+], correctly rounded
    double d = 0;
    const auto r = std::from_chars(s.data(), s.data() + s.size(), d, std::chars_format::general);
    if (r.ec == std::errc::result_out_of_range) { const std::string z(s); d = strtod(z.c_str(), nullptr); }   // inf / 0 / subnormal
    return d;
}

// Python float() on a cell that ascii_plain accepts: false where it raises, else *out = the value
static bool py_float(std::string_view v, double *out) {
    size_t a = 0, b = v.size();
    while (a < b && py_space((unsigned char)v[a])) a++;
    while (b > a && py_space((unsigned char)v[b - 1])) b--;
    if (a == b) return false;
    bool neg = false;
    if (v[a] == '+' || v[a] == '-') { neg = v[a] == '-'; a++; }
    const std::string_view s = v.substr(a, b - a);
    auto is = [&](const char *w) {
        const size_t n = strlen(w);
        if (s.size() != n) return false;
        for (size_t i = 0; i < n; i++) if ((s[i] | 0x20) != w[i]) return false;
        return true;
    };
    if (is("inf") || is("infinity")) { *out = neg ? -HUGE_VAL : HUGE_VAL; return true; }
    if (is("nan")) { *out = std::nan(""); return true; }
    size_t i = 0, nd = 0;
    while (i < s.size() && s[i] >= '0' && s[i] <= '9') { i++; nd++; }
    if (i < s.size() && s[i] == '.') { i++; while (i < s.size() && s[i] >= '0' && s[i] <= '9') { i++; nd++; } }
    if (!nd) return false;
    if (i < s.size() && (s[i] == 'e' || s[i] == 'E')) {
        i++;
        if (i < s.size() && (s[i] == '+' || s[i] == '-')) i++;
        size_t ne = 0;
        while (i < s.size() && s[i] >= '0' && s[i] <= '9') { i++; ne++; }
        if (!ne) return false;
    }
    if (i != s.size()) return false;
    const double d = parse_decimal(s);
    *out = neg ? -d : d;
    return true;
}

static double int_as_float(std::string_view v) {                // float(int(v)): correctly rounded, 0.0 for "-0"
    const IntText c = canon_int(v);
    if (c.digits.empty()) return 0.0;
    const double d = parse_decimal(c.digits);
    return c.neg ? -d : d;
}

// Python's repr(float): shortest round-trip digits, positional for exponents -4 .. 15, else d.ddde+XX
static void py_repr(double d, std::string &o) {
    if (std::isnan(d)) { o += "nan"; return; }
    if (std::isinf(d)) { o += d < 0 ? "-inf" : "inf"; return; }
    if (d == 0) { o += std::signbit(d) ? "-0.0" : "0.0"; return; }
    char buf[64];
    const auto r = std::to_chars(buf, buf + sizeof buf - 1, d, std::chars_format::scientific);
    *r.ptr = 0;
    const char *p = buf;
    if (*p == '-') { o += '-'; p++; }
    char dig[32];
    int nd = 0;
    for (; *p && *p != 'e'; p++) if (*p != '.') dig[nd++] = *p;
    const int ex = atoi(p + 1), decpt = ex + 1;
    if (decpt <= -4 || decpt > 16) {
        o += dig[0];
        if (nd > 1) { o += '.'; o.append(dig + 1, (size_t)nd - 1); }
        o += ex < 0 ? "e-" : "e+";
        const int ax = ex < 0 ? -ex : ex;
        if (ax < 10) o += '0';
        o += std::to_string(ax);
    } else if (decpt <= 0) {
        o += "0."; o.append((size_t)-decpt, '0'); o.append(dig, (size_t)nd);
    } else if (decpt >= nd) {
        o.append(dig, (size_t)nd); o.append((size_t)(decpt - nd), '0'); o += ".0";
    } else {
        o.append(dig, (size_t)decpt); o += '.'; o.append(dig + decpt, (size_t)(nd - decpt));
    }
}

// order-preserving key of a double; -0.0 and 0.0 are one value
static inline uint64_t float_key(double d) {
    if (d == 0) d = 0.0;
    uint64_t b;
    memcpy(&b, &d, 8);
    return (b >> 63) ? ~b : b | (1ull << 63);
}
constexpr uint64_t kNanKey0 = 0xFFF0000000000001ull;           // above +inf's key: NaN texts, in order of first appearance

template <class T, class Less>
static void sort_parallel(std::vector<T> &v, int P, Less less) {  // sorted chunks, then rounds of pairwise merges
    if (P <= 1 || v.size() < 100000) { std::sort(v.begin(), v.end(), less); return; }
    std::vector<size_t> b((size_t)P + 1);
    for (int k = 0; k <= P; k++) b[(size_t)k] = v.size() * (size_t)k / P;
    parallel_for(P, [&](int k) { std::sort(v.begin() + b[(size_t)k], v.begin() + b[(size_t)k + 1], less); });
    std::vector<T> tmp(v.size());
    for (int w = 1; w < P; w *= 2) {
        parallel_for((P + 2 * w - 1) / (2 * w), [&](int q) {
            const int k = q * 2 * w, mid = std::min(k + w, P), end = std::min(k + 2 * w, P);
            std::merge(v.begin() + b[(size_t)k], v.begin() + b[(size_t)mid], v.begin() + b[(size_t)mid], v.begin() + b[(size_t)end],
                       tmp.begin() + b[(size_t)k], less);
        });
        v.swap(tmp);
    }
}

// key[i] = rank of row i's cell among the column's distinct cells in byte order (Python's str order on UTF-8 text)
static void rank_strings(const std::string &t, const std::vector<uint64_t> &cell, std::vector<uint64_t> &key, int T) {
    const size_t n = cell.size();
    const int P = n < 200000 ? 1 : std::max(1, T);
    std::vector<std::vector<std::string_view>> local((size_t)P);
    parallel_for(P, [&](int p) {                                 // per piece: distinct cells, row -> local index
        std::unordered_map<std::string_view, uint32_t> seen;
        auto &L = local[(size_t)p];
        for (size_t i = n * (size_t)p / P, e = n * (size_t)(p + 1) / P; i < e; i++) {
            if (cell[i] == kSumAbsent) continue;
            const auto it = seen.emplace(cell_view(t, cell[i]), (uint32_t)L.size());
            if (it.second) L.push_back(it.first->first);
            key[i] = it.first->second;
        }
    });
    std::vector<std::string_view> all;
    for (auto &L : local) all.insert(all.end(), L.begin(), L.end());
    sort_parallel(all, P, std::less<std::string_view>());
    all.erase(std::unique(all.begin(), all.end()), all.end());
    parallel_for(P, [&](int p) {
        const auto &L = local[(size_t)p];
        std::vector<uint64_t> rank(L.size());
        for (size_t j = 0; j < L.size(); j++) rank[j] = (uint64_t)(std::lower_bound(all.begin(), all.end(), L[j]) - all.begin());
        for (size_t i = n * (size_t)p / P, e = n * (size_t)(p + 1) / P; i < e; i++)
            if (cell[i] != kSumAbsent) key[i] = rank[key[i]];
    });
}

// frontend._infer_column over one column, then the keys: equal typed values share a key, keys ascend in typed order
static void type_column(const std::string &t, SumColumn &C, int T) {
    const size_t n = C.cell.size();
    const int P = n < 100000 ? 1 : std::max(1, T);
    struct Seen { bool absent = false, not_int = false, not_float = false, long_int = false, nan = false; };
    std::vector<Seen> seen((size_t)P);
    parallel_for(P, [&](int p) {
        Seen &s = seen[(size_t)p];
        for (size_t i = n * (size_t)p / P, e = n * (size_t)(p + 1) / P; i < e; i++) {
            if (C.cell[i] == kSumAbsent) { s.absent = true; continue; }
            const std::string_view v = cell_view(t, C.cell[i]);
            if (strict_int(v)) { if (canon_int(v).digits.size() > 18) s.long_int = true; continue; }
            s.not_int = true;
            if (s.not_float) continue;
            double d;
            if (!ascii_plain(v) || !py_float(v, &d)) s.not_float = true;
            else if (d != d) s.nan = true;
        }
    });
    Seen all;
    for (auto &s : seen) { all.absent |= s.absent; all.not_int |= s.not_int; all.not_float |= s.not_float; all.long_int |= s.long_int; all.nan |= s.nan; }
    C.kind = !all.not_int ? (all.absent ? SUM_INT_AS_FLOAT : SUM_INT) : !all.not_float ? SUM_FLOAT : SUM_STRING;
    C.key.assign(n, kSumAbsent);
    if (C.kind == SUM_STRING) {
        rank_strings(t, C.cell, C.key, T);
    } else if (C.kind == SUM_INT && all.long_int) {             // ints beyond 64 bits: ranks of the canonical decimals
        std::unordered_map<std::string, uint64_t> id;
        std::vector<std::pair<bool, std::string_view>> uniq;
        auto txt = [](const IntText &c) { return std::string(c.neg ? "-" : "") + std::string(c.digits); };
        for (size_t i = 0; i < n; i++) {
            if (C.cell[i] == kSumAbsent) continue;
            const IntText c = canon_int(cell_view(t, C.cell[i]));
            if (id.emplace(txt(c), 0).second) uniq.emplace_back(c.neg, c.digits);
        }
        std::sort(uniq.begin(), uniq.end(), [](const auto &x, const auto &y) {
            if (x.first != y.first) return x.first;                  // negatives first
            const bool less_mag = x.second.size() != y.second.size() ? x.second.size() < y.second.size() : x.second < y.second;
            const bool more_mag = x.second.size() != y.second.size() ? x.second.size() > y.second.size() : y.second < x.second;
            return x.first ? more_mag : less_mag;
        });
        for (size_t r = 0; r < uniq.size(); r++) id[txt({uniq[r].first, uniq[r].second})] = r;
        for (size_t i = 0; i < n; i++) if (C.cell[i] != kSumAbsent) C.key[i] = id[txt(canon_int(cell_view(t, C.cell[i])))];
    } else {
        parallel_for(P, [&](int p) {
            for (size_t i = n * (size_t)p / P, e = n * (size_t)(p + 1) / P; i < e; i++) {
                if (C.cell[i] == kSumAbsent) continue;
                const std::string_view v = cell_view(t, C.cell[i]);
                if (C.kind == SUM_INT) {
                    const IntText c = canon_int(v);
                    int64_t x = 0;
                    for (char ch : c.digits) x = x * 10 + (ch - '0');
                    C.key[i] = (uint64_t)(c.neg ? -x : x) ^ (1ull << 63);
                } else {
                    double d = 0;
                    if (C.kind == SUM_INT_AS_FLOAT) d = int_as_float(v); else py_float(v, &d);
                    C.key[i] = d != d ? 0 : float_key(d);            // 0: a NaN, numbered below
                }
            }
        });
        if (all.nan) {                                           // one value per NaN text, as Python's float objects
            std::unordered_map<std::string_view, uint64_t> nan_id;
            for (size_t i = 0; i < n; i++)
                if (C.cell[i] != kSumAbsent && C.key[i] == 0) C.key[i] = kNanKey0 + nan_id.emplace(cell_view(t, C.cell[i]), nan_id.size()).first->second;
        }
    }
    uint64_t lo = ~0ull, hi = 0;
    for (size_t i = 0; i < n; i++) if (C.cell[i] != kSumAbsent) { lo = std::min(lo, C.key[i]); hi = std::max(hi, C.key[i]); }
    if (lo > hi) lo = hi = 0;
    for (size_t i = 0; i < n; i++) if (C.cell[i] != kSumAbsent) C.key[i] -= lo;
    C.bits = 1;
    while (C.bits < 64 && ((hi - lo) >> C.bits)) C.bits++;
}

void parse_summary_tsv(const std::string &path, const std::vector<std::string> &columns, SummaryTable &S, int threads) {
    slurp_maybe_gz(path, S.text);
    const std::string &t = S.text;
    if (t.size() >> 40) throw LimitError("per-read TSV of 1 TB or more");
    // header: the first line (CR, LF or CRLF ends a line, as in Python's text mode); the last of duplicate names wins
    size_t he = t.find_first_of("\r\n");
    if (he == std::string::npos) he = t.size();
    size_t body = he;
    if (body < t.size()) body += (t[body] == '\r' && body + 1 < t.size() && t[body + 1] == '\n') ? 2 : 1;
    auto rename = [](const std::string &h) -> std::string {       // convert_df_to_proper_umi :237
        if (h == "r1_CB") return "cb";
        if (h == "r1_UB") return "umi";
        if (h == "nimble_features") return "features";
        return h;
    };
    std::unordered_map<std::string, int> col;
    for (size_t a = 0, i = 0;; i++) {
        const size_t e = std::min(he, t.find('\t', a));
        col[rename(t.substr(a, e - a))] = (int)i;
        if (e >= he) break;
        a = e + 1;
    }
    std::vector<std::string> want{"umi"};
    for (auto &c : columns) want.push_back(rename(c));
    std::unordered_map<int, int> slot;                           // header index -> S.cols index
    for (size_t w = 0; w < want.size(); w++) {
        const auto it = col.find(want[w]);
        if (it == col.end()) throw MissingColumn(want[w]);
        auto s = slot.emplace(it->second, (int)S.cols.size());
        if (s.second) { S.cols.emplace_back(); S.cols.back().header_index = it->second; }
        if (w == 0) S.umi = s.first->second;
        else { S.out_cols.push_back(s.first->second); S.out_names.push_back(want[w]); }
    }
    const int K = (int)S.cols.size();
    std::vector<std::pair<int, int>> need;                       // (header index, cols index), ascending
    for (int k = 0; k < K; k++) need.emplace_back(S.cols[(size_t)k].header_index, k);
    std::sort(need.begin(), need.end());
    // body: pieces cut after LFs; inside a piece a lone CR also ends a line; short rows read empty (NA) cells
    const std::vector<size_t> cut = line_pieces(t, std::min(body, t.size()), threads);
    const int T = (int)cut.size() - 1;
    std::vector<std::vector<std::vector<uint64_t>>> parts((size_t)T, std::vector<std::vector<uint64_t>>((size_t)K));
    std::vector<uint64_t> rows((size_t)T, 0);
    parallel_for(T, [&](int k) {
        auto &P = parts[(size_t)k];
        size_t p = cut[(size_t)k];
        const size_t end = cut[(size_t)k + 1];
        uint64_t nr = 0;
        size_t e = 0;                                            // the next LF at or after p (end: none)
        bool e_ok = false;
        while (p < end) {
            if (!e_ok || e < p) {
                const void *nl = memchr(t.data() + p, '\n', end - p);
                e = nl ? (size_t)((const char *)nl - t.data()) : end;
                e_ok = true;
            }
            const void *cr = memchr(t.data() + p, '\r', e - p);
            size_t le = e, next = e + 1;
            if (cr) { le = (size_t)((const char *)cr - t.data()); next = (e < end && le + 1 == e) ? e + 1 : le + 1; }
            size_t a = p, q = 0;
            for (int f = 0; q < need.size(); f++) {
                const void *tb = memchr(t.data() + a, '\t', le - a);
                const size_t fe = tb ? (size_t)((const char *)tb - t.data()) : le;
                if (need[q].first == f) {
                    const std::string_view v(t.data() + a, fe - a);
                    if (v.size() >> 24) throw LimitError("a cell of 16 MB or more in the per-read TSV");
                    P[(size_t)need[q].second].push_back(pandas_na(v) ? kSumAbsent : ((uint64_t)a << 24) | v.size());
                    q++;
                }
                if (!tb) break;
                a = fe + 1;
            }
            for (; q < need.size(); q++) P[(size_t)need[q].second].push_back(kSumAbsent);
            nr++;
            p = next;
        }
        rows[(size_t)k] = nr;
    });
    std::vector<uint64_t> base((size_t)T + 1, 0);
    for (int k = 0; k < T; k++) base[(size_t)k + 1] = base[(size_t)k] + rows[(size_t)k];
    S.n_rows = base[(size_t)T];
    if (S.n_rows >= 0xFFFFFFFFull) throw LimitError("2^32 or more rows in the per-read TSV");
    for (int c = 0; c < K; c++) {
        auto &cell = S.cols[(size_t)c].cell;
        cell.resize(S.n_rows);
        parallel_for(T, [&](int k) {
            auto &v = parts[(size_t)k][(size_t)c];
            std::copy(v.begin(), v.end(), cell.begin() + (ptrdiff_t)base[(size_t)k]);
            std::vector<uint64_t>().swap(v);
        });
        type_column(t, S.cols[(size_t)c], threads);
    }
}

// Python's printed form of one typed cell
static void format_cell(const std::string &t, const SumColumn &C, uint32_t row, std::string &o) {
    const std::string_view v = cell_view(t, C.cell[row]);
    switch (C.kind) {
    case SUM_INT: { const IntText c = canon_int(v); if (c.digits.empty()) o += '0'; else { if (c.neg) o += '-'; o += c.digits; } break; }
    case SUM_INT_AS_FLOAT: py_repr(int_as_float(v), o); break;
    case SUM_FLOAT: { double d = 0; py_float(v, &d); py_repr(d, o); break; }
    case SUM_STRING: o += v; break;
    }
}

static void put_cell(std::string &o, const std::string &x) {     // csv.QUOTE_MINIMAL as pandas.to_csv applies it
    if (x.find_first_of("\t\"\r\n") == std::string::npos) { o += x; return; }
    o += '"';
    for (char ch : x) { if (ch == '"') o += '"'; o += ch; }
    o += '"';
}

void write_summary_tsv(const std::string &out_path, const SummaryTable &S, const std::vector<uint32_t> &umi_first,
                       const std::vector<SumRuns> &runs, int threads) {
    const std::string &t = S.text;
    const size_t U = umi_first.size();
    const int P = U < 20000 ? 1 : std::max(1, threads);
    std::vector<std::string> out((size_t)P);
    for (size_t j = 0; j < S.out_names.size() + 1; j++) {
        if (j) out[0] += '\t';
        put_cell(out[0], j ? S.out_names[j - 1] : std::string("umi"));
    }
    out[0] += '\n';
    parallel_for(P, [&](int p) {
        const uint32_t u0 = (uint32_t)(U * (size_t)p / P), u1 = (uint32_t)(U * (size_t)(p + 1) / P);
        std::vector<size_t> at;
        for (int c : S.out_cols) {
            const auto &R = runs[(size_t)c];
            at.push_back((size_t)(std::lower_bound(R.urank.begin(), R.urank.end(), u0) - R.urank.begin()));
        }
        std::string &o = out[(size_t)p], x;
        for (uint32_t u = u0; u < u1; u++) {
            x.clear();
            format_cell(t, S.cols[(size_t)S.umi], umi_first[u], x);
            put_cell(o, x);
            for (size_t j = 0; j < S.out_cols.size(); j++) {
                const int c = S.out_cols[j];
                const auto &R = runs[(size_t)c];
                x.clear();
                for (size_t &i = at[j]; i < R.urank.size() && R.urank[i] == u; i++) {
                    if (!x.empty()) x += "; ";
                    format_cell(t, S.cols[(size_t)c], R.first[i], x);
                    x += '('; x += std::to_string(R.count[i]); x += ')';
                }
                o += '\t';
                put_cell(o, x);
            }
            o += '\n';
        }
    });
    const std::string tmp = out_path + ".tmp";
    FILE *f = fopen(tmp.c_str(), "wb");
    if (!f) throw IoError("cannot write " + tmp);
    for (auto &s : out)
        if (!s.empty() && fwrite(s.data(), 1, s.size(), f) != s.size()) { fclose(f); throw IoError("write failed on " + tmp); }
    if (fclose(f) != 0) throw IoError("close failed on " + tmp);
    if (rename(tmp.c_str(), out_path.c_str()) != 0) throw IoError("cannot rename " + tmp);
}

}  // namespace nb200

using namespace nb200;

extern "C" int32_t nb200_summary_cell_type(const char *cell, uint64_t len, double *value) {
    if (!cell && len) return NB200_EINVAL;
    const std::string_view v(cell ? cell : "", (size_t)len);
    double d = 0;
    int32_t kind = 3;
    if (pandas_na(v)) kind = 0;
    else if (strict_int(v)) { kind = 1; d = int_as_float(v); }
    else if (ascii_plain(v) && py_float(v, &d)) kind = 2;
    if (value) *value = d;
    return kind;
}

extern "C" int32_t nb200_float_repr(double x, char *out, int32_t cap) {
    std::string s;
    py_repr(x, s);
    if (!out || cap <= (int32_t)s.size()) return NB200_EINVAL;
    memcpy(out, s.data(), s.size());
    out[s.size()] = 0;
    return (int32_t)s.size();
}
