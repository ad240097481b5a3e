// Library JSON -> host images of the GPU index (SURVEY.md §8a rows A1, A2, X1).
#include "library.hpp"

#include <algorithm>
#include <atomic>
#include <cerrno>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <numeric>
#include <sstream>
#include <stdexcept>
#include <thread>
#include <unordered_map>

#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include "checksum.hpp"
#include "ingest.hpp"
#include "json.hpp"
#include "kmer_hash.hpp"

namespace nb200 {

uint64_t hash_kmer(uint64_t x) {       // identical to dev_hash_kmer (kernels.cuh)
    x ^= x >> 29;
    x *= 0xD6E8FEB86659FD93ull;
    x ^= x >> 32;
    return x;
}

uint64_t revcomp_kmer(uint64_t x, int k) {
    uint64_t y = ~x;                                   // complement, then reverse the 2-bit groups
    y = ((y >> 2) & 0x3333333333333333ull) | ((y & 0x3333333333333333ull) << 2);
    y = ((y >> 4) & 0x0F0F0F0F0F0F0F0Full) | ((y & 0x0F0F0F0F0F0F0F0Full) << 4);
    y = __builtin_bswap64(y);
    return y >> (64 - 2 * k);
}

int parse_strand_filter(const char *s) {
    if (!s || !*s) return NB200_UNSTRANDED;
    std::string v(s);
    if (v == "unstranded") return NB200_UNSTRANDED;
    if (v == "fiveprime") return NB200_FIVEPRIME;
    if (v == "threeprime") return NB200_THREEPRIME;
    if (v == "none") return NB200_STRAND_NONE;
    return -1;
}

static int cfg_int(const JValue &c, const char *key, int dflt) {
    const JValue *v = c.get(key);
    if (!v) return dflt;
    if (v->type == JValue::Num) return (int)v->num;
    if (v->type == JValue::Bool) return v->b ? 1 : 0;
    return dflt;
}

static double cfg_num(const JValue &c, const char *key, double dflt) {
    const JValue *v = c.get(key);
    return (v && v->type == JValue::Num) ? v->num : dflt;
}

void parse_library_json(const std::string &path, std::vector<std::string> &names, std::vector<std::string> &seqs,
                        std::vector<std::string> &features, nb200_config &cfg) {
    std::ifstream f(path, std::ios::binary);
    if (!f) throw std::runtime_error("cannot open library file " + path);
    std::stringstream ss;
    ss << f.rdbuf();
    std::string text = ss.str();
    JValue root = JParser(text.data(), text.size()).parse();
    if (root.type != JValue::Arr || root.arr.size() < 2 || root.arr[0].type != JValue::Obj ||
        root.arr[1].type != JValue::Obj)
        throw std::runtime_error("library JSON must be [config, data] (nimble/__main__.py:64-65)");
    const JValue &c = root.arr[0], &d = root.arr[1];
    // defaults = nimble/types.py:12-25
    cfg.score_threshold = cfg_int(c, "score_threshold", 20);
    cfg.score_filter = cfg_int(c, "score_filter", 25);
    cfg.score_percent = cfg_num(c, "score_percent", 0.5);
    cfg.num_mismatches = cfg_int(c, "num_mismatches", 0);
    cfg.discard_multiple_matches = cfg_int(c, "discard_multiple_matches", 0);
    cfg.intersect_level = cfg_int(c, "intersect_level", 0);
    cfg.discard_multi_hits = cfg_int(c, "discard_multi_hits", 0);
    cfg.require_valid_pair = cfg_int(c, "require_valid_pair", 0);
    cfg.max_hits_to_report = cfg_int(c, "max_hits_to_report", 10);
    std::string group_on;
    if (const JValue *g = c.get("group_on"); g && g->type == JValue::Str) group_on = g->str;

    const JValue *h = d.get("headers"), *cols = d.get("columns");
    if (!h || !cols || h->type != JValue::Arr || cols->type != JValue::Arr || h->arr.size() != cols->arr.size())
        throw std::runtime_error("library data needs matching 'headers' and 'columns' (nimble/types.py:29-32)");
    int i_name = -1, i_seq = -1, i_group = -1;
    for (size_t i = 0; i < h->arr.size(); i++) {
        const std::string &s = h->arr[i].str;
        if (s == "sequence_name") i_name = (int)i;
        else if (s == "sequence") i_seq = (int)i;
        if (!group_on.empty() && s == group_on) i_group = (int)i;
    }
    if (i_name < 0 || i_seq < 0) throw std::runtime_error("library data lacks sequence_name / sequence columns");
    const JValue &cn = cols->arr[i_name], &cs = cols->arr[i_seq];
    if (cn.type != JValue::Arr || cs.type != JValue::Arr || cn.arr.size() != cs.arr.size())
        throw std::runtime_error("library columns have different lengths");
    const JValue *cg = i_group >= 0 ? &cols->arr[i_group] : nullptr;
    if (cg && (cg->type != JValue::Arr || cg->arr.size() != cn.arr.size()))
        throw std::runtime_error("group_on column has a different length");
    size_t n = cn.arr.size();
    names.resize(n); seqs.resize(n); features.resize(n);
    for (size_t i = 0; i < n; i++) {
        names[i] = cn.arr[i].str;
        seqs[i] = cs.arr[i].str;
        features[i] = cg ? cg->arr[i].str : names[i];
    }
}

static void token_ranks(const std::vector<std::string> &names, std::vector<uint32_t> &te, std::vector<uint32_t> &tc) {
    // Order of the comma-joined feature strings pandas sorts by (nimble/__main__.py:248-251,289)
    // == lexicographic order of token sequences, token = name + ',' (inner) or name + NUL (last).
    size_t F = names.size();
    struct Tok { std::string s; uint32_t id; uint8_t kind; };
    std::vector<Tok> toks;
    toks.reserve(2 * F);
    for (size_t i = 0; i < F; i++) {
        toks.push_back({names[i] + std::string(1, '\0'), (uint32_t)i, 0});
        toks.push_back({names[i] + ",", (uint32_t)i, 1});
    }
    std::sort(toks.begin(), toks.end(), [](const Tok &a, const Tok &b) {
        int c = memcmp(a.s.data(), b.s.data(), std::min(a.s.size(), b.s.size()));
        if (c) return c < 0;
        return a.s.size() < b.s.size();
    });
    te.assign(F, 0); tc.assign(F, 0);
    for (size_t r = 0; r < toks.size(); r++) (toks[r].kind ? tc : te)[toks[r].id] = (uint32_t)r;
}

static bool bytes_less(const std::string &a, const std::string &b) {
    int c = memcmp(a.data(), b.data(), std::min(a.size(), b.size()));
    if (c) return c < 0;
    return a.size() < b.size();
}

void build_feature_dictionary(const std::vector<std::string> &sorted_names, HostLibrary &out) {
    for (size_t i = 0; i < sorted_names.size(); i++) {
        const std::string &s = sorted_names[i];
        if (s.find(',') != std::string::npos || s.find('\t') != std::string::npos || s.find('\n') != std::string::npos ||
            s.find('\0') != std::string::npos)
            throw std::runtime_error("feature name contains ',', TAB, NUL or newline: " + s);
        if (i && !bytes_less(sorted_names[i - 1], s)) throw std::runtime_error("feature names must be sorted and unique");
    }
    out.feature_names = sorted_names;
    out.n_features = (uint32_t)sorted_names.size();
    token_ranks(sorted_names, out.tok_end, out.tok_comma);
}

static inline int base_code(char c) {
    switch (c) {
    case 'A': case 'a': return 0;
    case 'C': case 'c': return 1;
    case 'G': case 'g': return 2;
    case 'T': case 't': return 3;
    default: return 4;
    }
}

struct Occ { uint64_t kmer; uint32_t ref, pos; };

template <class F>
static void parallel_for(int T, size_t n, F f) {      // f(thread, begin, end) over [0, n)
    if (T <= 1 || n < 4096) { f(0, (size_t)0, n); return; }
    std::vector<std::thread> th;
    const size_t per = (n + T - 1) / T;
    for (int t = 0; t < T; t++) {
        const size_t a = std::min(n, t * per), b = std::min(n, a + per);
        if (a < b) th.emplace_back([=] { f(t, a, b); });
    }
    for (auto &x : th) x.join();
}

// Sort records by a 64-bit key whose top `key_bits` bits are significant: one counting pass into
// 256 buckets on the top 8 bits, then the buckets are sorted independently on T threads.
template <class Rec, class KeyOf, class Less>
static void bucket_sort(std::vector<Rec> &v, int key_bits, int T, KeyOf key_of, Less less) {
    const size_t n = v.size();
    if (n < (1u << 16) || T <= 1) { std::sort(v.begin(), v.end(), less); return; }
    const int shift = key_bits > 8 ? key_bits - 8 : 0;
    std::vector<size_t> cnt((size_t)T * 256, 0);
    parallel_for(T, n, [&](int t, size_t a, size_t b) {
        size_t *c = &cnt[(size_t)t * 256];
        for (size_t i = a; i < b; i++) c[(key_of(v[i]) >> shift) & 255]++;
    });
    std::vector<size_t> start(257, 0), off((size_t)T * 256, 0);
    size_t run = 0;
    for (int bkt = 0; bkt < 256; bkt++) {
        start[bkt] = run;
        for (int t = 0; t < T; t++) { off[(size_t)t * 256 + bkt] = run; run += cnt[(size_t)t * 256 + bkt]; }
    }
    start[256] = run;
    std::vector<Rec> out(n);
    parallel_for(T, n, [&](int t, size_t a, size_t b) {      // same partition as the counting pass
        size_t *o = &off[(size_t)t * 256];
        for (size_t i = a; i < b; i++) out[o[(key_of(v[i]) >> shift) & 255]++] = v[i];
    });
    v.swap(out);
    std::vector<Rec>().swap(out);
    std::atomic<int> next{0};
    std::vector<std::thread> th;
    for (int t = 0; t < T; t++)
        th.emplace_back([&] {
            for (int bkt; (bkt = next.fetch_add(1)) < 256;) std::sort(v.begin() + start[bkt], v.begin() + start[bkt + 1], less);
        });
    for (auto &x : th) x.join();
}

// One table lookup as the GPU does it (probe_lookup in kernels.cuh): read k-mer x -> class / position offset of the
// library k-mers equal to x (cl[0], read as sequenced) and to revcomp(x) (cl[1], read reverse-complemented).
void host_lookup(const HostLibrary &L, uint64_t x, uint32_t cl[2], uint32_t of[2]) {
    const int k = L.cfg.k;
    const uint64_t y = revcomp_kmer(x, k), c = x < y ? x : y;
    const uint32_t nb = (uint32_t)L.n_buckets, mix = kmer_mix((uint32_t)c, (uint32_t)(c >> 32));
    const uint32_t b1 = kmer_bucket1(mix, nb);
    const Entry *e = nullptr;
    const Entry *bk = &L.table[2 * (size_t)b1];
    if (bk[0].key == c) e = &bk[0]; else if (bk[1].key == c) e = &bk[1];
    if (!e && (bk[0].cls & kClsSpill)) {
        const uint32_t b2 = kmer_bucket2(mix, (uint32_t)c, b1, nb);
        bk = &L.table[2 * (size_t)b2];
        if (bk[0].key == c) e = &bk[0]; else if (bk[1].key == c) e = &bk[1];
    }
    cl[0] = cl[1] = kEmptyClass; of[0] = of[1] = 0;
    if (!e) return;
    uint32_t cls_s = kEmptyClass, off_s = 0, cls_r = kEmptyClass, off_r = 0;
    if (e->cls & kClsDual) { const DualRec &d = L.dual[e->cls & kClsIdMask]; cls_s = d.cls_s; off_s = d.off_s; cls_r = d.cls_r; off_r = d.off_r; }
    else if (e->cls & kClsRc) { cls_r = e->cls & kClsIdMask; off_r = e->off; }
    else { cls_s = e->cls & kClsIdMask; off_s = e->off; }
    const bool xs = x == c, ys = y == c;
    cl[0] = xs ? cls_s : cls_r; of[0] = xs ? off_s : off_r;
    cl[1] = ys ? cls_s : cls_r; of[1] = ys ? off_s : off_r;
}

void build_library(const std::vector<std::string> &names, const std::vector<std::string> &seqs,
                   const std::vector<std::string> &features, const nb200_config &cfg, int host_threads,
                   HostLibrary &L, bool verify) {
    const bool timing = getenv("NB200_BUILD_TIMING") != nullptr;
    auto t_last = std::chrono::steady_clock::now();
    auto lap = [&](const char *what) {
        if (!timing) return;
        auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "[nb200 build] %-28s %.2f s\n", what, std::chrono::duration<double>(now - t_last).count());
        t_last = now;
    };
    const int k = cfg.k;
    if (k < 4 || k > 32) throw std::runtime_error("k must be in 4..32");
    if (cfg.max_hits_to_report < 1 || cfg.max_hits_to_report > 64)
        throw LimitError("max_hits_to_report must be in 1..64");
    if (cfg.strand_filter < 0 || cfg.strand_filter > 3) throw std::runtime_error("bad strand_filter");
    const size_t R = names.size();
    if (seqs.size() != R || features.size() != R) throw std::runtime_error("names/seqs/features differ in length");
    if (R == 0) throw std::runtime_error("library has no sequences");
    if (R > kMaxRefs) throw LimitError("library has more than 2,097,120 sequences (16-bit class word index)");
    L.cfg = cfg;
    // ---- features: id = rank of the name in byte order ------------------------------------------
    std::vector<std::string> fn(features);
    std::sort(fn.begin(), fn.end(), bytes_less);
    fn.erase(std::unique(fn.begin(), fn.end()), fn.end());
    build_feature_dictionary(fn, L);
    std::vector<uint32_t> fid(R);
    for (size_t i = 0; i < R; i++)
        fid[i] = (uint32_t)(std::lower_bound(fn.begin(), fn.end(), features[i], bytes_less) - fn.begin());
    // ---- internal reference order: (feature id, input order) ------------------------------------
    std::vector<uint32_t> order(R);
    std::iota(order.begin(), order.end(), 0u);
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return fid[a] < fid[b]; });
    L.n_refs = (uint32_t)R;
    L.ref_names.resize(R); L.ref_feature.resize(R); L.ref_len.resize(R); L.ref_gstart.resize(R);
    L.identity_features = (L.n_features == R);
    uint64_t g = kRefPad;
    for (size_t r = 0; r < R; r++) {
        uint32_t src = order[r];
        L.ref_names[r] = names[src];
        L.ref_feature[r] = fid[src];
        if (fid[src] != r) L.identity_features = false;
        L.ref_len[r] = (uint32_t)seqs[src].size();
        if (g + seqs[src].size() + kRefPad + 128 >= 0xFFFFFFFFull) throw LimitError("library exceeds 4 Gbases");
        L.ref_gstart[r] = (uint32_t)g;
        g += seqs[src].size() + kRefPad;
    }
    L.total_gbases = g + 128;
    const size_t n_words = (size_t)((L.total_gbases + 31) / 32) + 2;
    L.ref2bit.assign(n_words, 0);
    L.refN.assign(n_words, 0xFFFFFFFFu);
    // ---- k-mer occurrences (threads own disjoint reference ranges; padding keeps their words apart) ----
    const int T = std::max(1, host_threads);
    const uint64_t kmask = k == 32 ? ~0ull : ((1ull << (2 * k)) - 1);
    std::vector<Occ> occ;
    {
        std::vector<size_t> first(R + 1, 0);
        for (size_t r = 0; r < R; r++) first[r + 1] = first[r] + (L.ref_len[r] >= (uint32_t)k ? L.ref_len[r] - k + 1 : 0);
        occ.resize(first[R]);
        parallel_for(T, R, [&](int, size_t ra, size_t rb) {
            for (size_t r = ra; r < rb; r++) {
                const std::string &s = seqs[order[r]];
                uint64_t x = 0; int valid = 0;
                const uint64_t g0 = L.ref_gstart[r];
                size_t w = first[r];
                for (size_t i = 0; i < s.size(); i++) {
                    int c = base_code(s[i]);
                    if (c > 3) { valid = 0; x = 0; continue; }
                    uint64_t gp = g0 + i;
                    L.ref2bit[gp >> 5] |= (uint64_t)c << (2 * (gp & 31));
                    L.refN[gp >> 5] &= ~(1u << (gp & 31));
                    x = ((x >> 2) | ((uint64_t)c << (2 * (k - 1)))) & kmask;
                    if (++valid >= k) occ[w++] = Occ{x, (uint32_t)r, (uint32_t)(i + 1 - k)};
                }
                for (; w < first[r + 1]; w++) occ[w] = Occ{~0ull, 0xFFFFFFFFu, 0};   // k-mers lost to non-ACGT bases
            }
        });
    }
    bucket_sort(occ, 2 * k, T, [](const Occ &o) { return o.kmer; }, [](const Occ &a, const Occ &b) {
        if (a.kmer != b.kmer) return a.kmer < b.kmer;
        if (a.ref != b.ref) return a.ref < b.ref;
        return a.pos < b.pos;
    });
    while (!occ.empty() && occ.back().ref == 0xFFFFFFFFu) occ.pop_back();   // fillers sort last (key all ones)
    lap("occurrences + sort");
    // ---- distinct k-mers -> member lists (ascending ref) + first positions ---------------------
    std::vector<uint64_t> kmers;
    std::vector<uint64_t> mem_off;     // per k-mer, into mem_ref / positions
    std::vector<uint32_t> mem_ref;
    L.positions.clear();
    {
        size_t nk = 0;
        for (size_t i = 0; i < occ.size(); i++) nk += (i == 0 || occ[i].kmer != occ[i - 1].kmer);
        kmers.reserve(nk); mem_off.reserve(nk + 1); mem_ref.reserve(occ.size()); L.positions.reserve(occ.size());
    }
    for (size_t i = 0; i < occ.size(); i++) {
        bool newk = (i == 0 || occ[i].kmer != occ[i - 1].kmer);
        if (newk) { kmers.push_back(occ[i].kmer); mem_off.push_back(mem_ref.size()); }
        if (newk || occ[i].ref != occ[i - 1].ref) { mem_ref.push_back(occ[i].ref); L.positions.push_back(occ[i].pos); }
    }
    mem_off.push_back(mem_ref.size());
    if (mem_ref.size() >= 0xFFFFFFFFull) throw LimitError("more than 4 G k-mer occurrences");
    std::vector<Occ>().swap(occ);
    L.n_kmers = kmers.size();
    lap("distinct k-mers");
    // ---- equivalence classes = distinct member lists --------------------------------------------
    std::vector<uint32_t> kclass(kmers.size());
    std::vector<uint64_t> class_rep;   // representative k-mer index per class
    {
        std::unordered_map<uint64_t, std::vector<uint32_t>> by_hash;
        by_hash.reserve(std::min<size_t>(kmers.size() / 4 + 16, 1u << 22));
        std::vector<uint32_t> single(R, kEmptyClass);        // classes with exactly one member: no hashing
        for (size_t q = 0; q < kmers.size(); q++) {
            uint64_t a = mem_off[q], b = mem_off[q + 1];
            if (b - a == 1) {
                uint32_t &c1 = single[mem_ref[a]];
                if (c1 == kEmptyClass) { c1 = (uint32_t)class_rep.size(); class_rep.push_back(q); }
                kclass[q] = c1;
                continue;
            }
            uint64_t h = 0x9E3779B97F4A7C15ull ^ (b - a);
            for (uint64_t j = a; j < b; j++) h = hash_kmer(h ^ mem_ref[j]);
            auto &bucket = by_hash[h];
            uint32_t found = kEmptyClass;
            for (uint32_t c : bucket) {
                uint64_t ra = mem_off[class_rep[c]], rb = mem_off[class_rep[c] + 1];
                if (rb - ra == b - a && memcmp(&mem_ref[ra], &mem_ref[a], (b - a) * sizeof(uint32_t)) == 0) { found = c; break; }
            }
            if (found == kEmptyClass) {
                found = (uint32_t)class_rep.size();
                class_rep.push_back(q);
                bucket.push_back(found);
            }
            kclass[q] = found;
        }
    }
    L.n_classes = class_rep.size();
    lap("class dedup");
    L.n_words = (uint32_t)((R + 31) / 32);
    L.class_rec.assign(L.n_classes, ClassRec{});
    L.ov_w.clear(); L.ov_b.clear(); L.ov_pre.clear();
    for (size_t c = 0; c < class_rep.size(); c++) {
        std::vector<std::pair<uint32_t, uint32_t>> pairs;     // members are ascending
        for (uint64_t j = mem_off[class_rep[c]]; j < mem_off[class_rep[c] + 1]; j++) {
            const uint32_t w = mem_ref[j] >> 5, bit = 1u << (mem_ref[j] & 31);
            if (pairs.empty() || pairs.back().first != w) pairs.emplace_back(w, bit);
            else pairs.back().second |= bit;
        }
        ClassRec &rec = L.class_rec[c];
        uint32_t w[kRecInline];
        for (int i = 0; i < kRecInline; i++) { w[i] = kNoWord; rec.b[i] = 0; }
        rec.spare = 0;
        if (pairs.size() <= (size_t)kRecInline) {
            for (size_t i = 0; i < pairs.size(); i++) { w[i] = pairs[i].first; rec.b[i] = pairs[i].second; }
            rec.meta = (uint32_t)pairs.size();
        } else {
            if (L.ov_w.size() + pairs.size() >= 0xFFFFFFFFull) throw LimitError("class overflow table exceeds 4 G pairs");
            rec.meta = kRecOverflow;
            rec.b[0] = (uint32_t)L.ov_w.size();
            rec.b[1] = (uint32_t)pairs.size();
            uint32_t pre = 0;
            for (auto &pr : pairs) {
                L.ov_w.push_back(pr.first); L.ov_b.push_back(pr.second); L.ov_pre.push_back(pre);
                pre += (uint32_t)__builtin_popcount(pr.second);
            }
        }
        rec.w01 = w[0] | (w[1] << 16); rec.w23 = w[2] | (w[3] << 16);
    }
    lap("class records");
    if (L.n_classes > kClsIdMask) throw LimitError("more than 2^29 equivalence classes");
    // ---- canonical k-mer table (bucketed cuckoo, see library.hpp) -----------------------------------
    // 1. which canonical keys exist, and on which strand(s): k-mers are sorted, so the partner of a
    //    non-canonical k-mer is found by binary search.  owner[q] = 1: k-mer q creates the entry.
    const size_t nk = kmers.size();
    std::vector<uint8_t> role(nk);          // 0 entry with own-strand info, 1 entry with rc info, 2 dual entry, 3 covered by its partner
    std::vector<uint32_t> partner(nk, 0);
    parallel_for(T, nk, [&](int, size_t qa, size_t qb) {
        for (size_t q = qa; q < qb; q++) {
            const uint64_t x = kmers[q], y = revcomp_kmer(x, k);
            if (x == y) { role[q] = 0; continue; }                       // palindrome: own strand
            const auto it = std::lower_bound(kmers.begin(), kmers.end(), y);
            const bool has = it != kmers.end() && *it == y;
            if (x < y) { role[q] = has ? 2 : 0; if (has) partner[q] = (uint32_t)(it - kmers.begin()); }
            else role[q] = has ? 3 : 1;
        }
    });
    L.dual.clear();
    size_t n_keys = 0;
    for (size_t q = 0; q < nk; q++) {
        if (role[q] == 3) continue;
        n_keys++;
        if (role[q] == 2) {
            const size_t r = partner[q];
            partner[q] = (uint32_t)L.dual.size();
            L.dual.push_back(DualRec{kclass[q], (uint32_t)mem_off[q], kclass[r], (uint32_t)mem_off[r]});
        }
    }
    if (L.dual.size() > kClsIdMask) throw LimitError("more than 2^29 k-mers present on both strands");
    // 2. size: load factor = keys / entries; NB200_TABLE_LF overrides (tests force dense tables)
    // small tables (<= 256 MB) are built sparse: 1.5 % of the buckets spill instead of 8 %, so most probe rounds skip the
    // second-bucket path altogether
    double lf = n_keys <= (4u << 20) ? 0.25 : 0.5;
    if (const char *e = getenv("NB200_TABLE_LF")) lf = std::min(0.95, std::max(0.02, atof(e)));
    for (int attempt = 0;; attempt++) {
        uint64_t nb = (uint64_t)((double)n_keys / (2.0 * lf)) + 2;
        if (nb >= 0xFFFFFFFFull) throw LimitError("k-mer table exceeds 4 G buckets");
        L.n_buckets = nb;
        Entry empty{kEmptyKey, 0, 0};
        L.table.assign(2 * nb, empty);
        Entry *tab = L.table.data();
        auto buckets_of = [&](uint64_t canon, uint32_t &b1, uint32_t &b2) {
            const uint32_t mix = kmer_mix((uint32_t)canon, (uint32_t)(canon >> 32));
            b1 = kmer_bucket1(mix, (uint32_t)nb);
            b2 = kmer_bucket2(mix, (uint32_t)canon, b1, (uint32_t)nb);
        };
        auto entry_of = [&](size_t q) {
            const uint64_t x = kmers[q];
            Entry e;
            e.key = role[q] == 1 ? revcomp_kmer(x, k) : x;
            if (role[q] == 2) { e.cls = kClsDual | partner[q]; e.off = 0; }
            else { e.cls = kclass[q] | (role[q] == 1 ? kClsRc : 0u); e.off = (uint32_t)mem_off[q]; }
            return e;
        };
        // 3. lock-free first pass: claim a free entry of b1, else of b2 (CAS on the key); the rest waits
        std::vector<std::vector<uint32_t>> left(T);
        parallel_for(T, nk, [&](int t, size_t qa, size_t qb) {
            for (size_t q = qa; q < qb; q++) {
                if (role[q] == 3) continue;
                const Entry e = entry_of(q);
                uint32_t b[2];
                buckets_of(e.key, b[0], b[1]);
                bool placed = false;
                for (int c = 0; c < 4 && !placed; c++) {
                    Entry &slot = tab[2 * (size_t)b[c >> 1] + (c & 1)];
                    uint64_t expect = kEmptyKey;
                    if (__atomic_load_n(&slot.key, __ATOMIC_RELAXED) == kEmptyKey &&
                        __atomic_compare_exchange_n(&slot.key, &expect, e.key, false, __ATOMIC_ACQ_REL, __ATOMIC_ACQUIRE)) {
                        slot.cls = e.cls; slot.off = e.off;
                        placed = true;
                    }
                }
                if (!placed) left[t].push_back((uint32_t)q);
            }
        });
        // 4. the few keys whose four entries were taken: sequential random-walk cuckoo insertion
        bool ok = true;
        uint64_t rng = 0x9E3779B97F4A7C15ull;
        for (int t = 0; t < T && ok; t++)
            for (uint32_t q : left[t]) {
                Entry cur = entry_of(q);
                uint32_t avoid = 0xFFFFFFFFu;
                int kicks = 0;
                for (; kicks < 2000; kicks++) {
                    uint32_t b[2];
                    buckets_of(cur.key, b[0], b[1]);
                    bool placed = false;
                    for (int c = 0; c < 4 && !placed; c++) {
                        Entry &slot = tab[2 * (size_t)b[c >> 1] + (c & 1)];
                        if (slot.key == kEmptyKey) { slot = cur; placed = true; }
                    }
                    if (placed) break;
                    rng = hash_kmer(rng + kicks + 1);
                    uint32_t vb = b[(rng >> 7) & 1];
                    if (vb == avoid) vb = b[0] == avoid ? b[1] : b[0];      // do not bounce straight back
                    Entry &victim = tab[2 * (size_t)vb + ((rng >> 9) & 1)];
                    std::swap(cur, victim);
                    avoid = vb;
                }
                if (kicks == 2000) { ok = false; break; }
            }
        if (!ok) {                                   // cannot happen at sane load factors; thin the table out and redo
            if (attempt >= 6) throw std::runtime_error("k-mer table construction failed");
            lf *= 0.8;
            continue;
        }
        // 5. spill bits + statistics
        std::atomic<uint64_t> spilled{0};
        parallel_for(T, (size_t)nb, [&](int, size_t ba, size_t bb) {
            uint64_t sp = 0;
            for (size_t bkt = ba; bkt < bb; bkt++)
                for (int c = 0; c < 2; c++) {
                    const Entry &e = tab[2 * bkt + c];
                    if (e.key == kEmptyKey) continue;
                    uint32_t b1, b2;
                    buckets_of(e.key, b1, b2);
                    if (b1 != bkt) { __atomic_fetch_or(&tab[2 * (size_t)b1].cls, kClsSpill, __ATOMIC_RELAXED); sp++; }
                }
            spilled += sp;
        });
        L.n_spilled = spilled;
        break;
    }
    lap("table insertion");
    L.has_index = true;
    if (verify) {
        // every library k-mer, read in either orientation, must come back with its class and position offset; k-mers
        // that are not in the library must miss.  Same protocol as probe_lookup (kernels.cuh).
        std::atomic<uint64_t> bad{0};
        parallel_for(T, nk, [&](int, size_t qa, size_t qb) {
            uint64_t rng = 0x1234567ull + qa;
            for (size_t q = qa; q < qb; q++) {
                const uint64_t x = kmers[q], y = revcomp_kmer(x, k);
                const auto it = std::lower_bound(kmers.begin(), kmers.end(), y);
                const bool has = it != kmers.end() && *it == y;
                uint32_t cl[2], of[2];
                host_lookup(L, x, cl, of);
                bool ok = cl[0] == kclass[q] && of[0] == (uint32_t)mem_off[q];
                if (has) { const size_t r = (size_t)(it - kmers.begin()); ok = ok && cl[1] == kclass[r] && of[1] == (uint32_t)mem_off[r]; }
                else ok = ok && cl[1] == kEmptyClass;
                rng = hash_kmer(rng + q);
                const uint64_t z = rng & kmask;                          // a random k-mer: almost surely absent
                const uint64_t zr = revcomp_kmer(z, k);
                const bool zin = std::binary_search(kmers.begin(), kmers.end(), z), zrin = std::binary_search(kmers.begin(), kmers.end(), zr);
                host_lookup(L, z, cl, of);
                ok = ok && (cl[0] != kEmptyClass) == zin && (cl[1] != kEmptyClass) == zrin;
                if (!ok) bad++;
            }
        });
        if (bad) throw std::runtime_error("k-mer table self-check failed for " + std::to_string((uint64_t)bad) + " k-mers");
        lap("table self-check");
    }
}

// ---- device image -------------------------------------------------------------------------------------------------

ImageLayout image_layout(const uint64_t bytes[kImageParts]) {
    ImageLayout lay;
    for (int p = 0; p < kImageParts; p++) {
        lay.bytes[p] = bytes[p];
        lay.off[p] = lay.total;
        lay.total += ((bytes[p] + 255) & ~(uint64_t)255) + 256;
    }
    return lay;
}

struct PartSrc { const void *p; uint64_t bytes; };
static void image_parts(const HostLibrary &L, PartSrc out[kImageParts]) {
    auto v = [](const auto &vec) { return PartSrc{vec.data(), (uint64_t)vec.size() * sizeof(vec[0])}; };
    out[kPartTable] = v(L.table); out[kPartClassRec] = v(L.class_rec);
    out[kPartOvW] = v(L.ov_w); out[kPartOvB] = v(L.ov_b); out[kPartOvPre] = v(L.ov_pre);
    out[kPartPositions] = v(L.positions); out[kPartRefGstart] = v(L.ref_gstart); out[kPartRefFeature] = v(L.ref_feature);
    out[kPartRef2bit] = v(L.ref2bit); out[kPartRefN] = v(L.refN); out[kPartDual] = v(L.dual);
}

ImageLayout image_layout(const HostLibrary &L) {
    PartSrc src[kImageParts];
    image_parts(L, src);
    uint64_t bytes[kImageParts];
    for (int p = 0; p < kImageParts; p++) bytes[p] = src[p].bytes;
    return image_layout(bytes);
}

void image_fill(const HostLibrary &L, const ImageLayout &lay, uint64_t offset, uint64_t len, uint8_t *dst) {
    PartSrc src[kImageParts];
    image_parts(L, src);
    memset(dst, 0, len);
    for (int p = 0; p < kImageParts; p++) {
        const uint64_t a = std::max(offset, lay.off[p]), b = std::min(offset + len, lay.off[p] + lay.bytes[p]);
        if (a < b) memcpy(dst + (a - offset), static_cast<const uint8_t *>(src[p].p) + (a - lay.off[p]), b - a);
    }
}

HostLibrary library_meta(const HostLibrary &L) {
    HostLibrary m;
    m.cfg = L.cfg; m.has_index = L.has_index;
    m.trim_on = L.trim_on; m.trim_target = L.trim_target; m.trim_strictness = L.trim_strictness;
    m.feature_names = L.feature_names; m.tok_end = L.tok_end; m.tok_comma = L.tok_comma;
    m.ref_names = L.ref_names; m.ref_feature = L.ref_feature; m.ref_len = L.ref_len; m.ref_gstart = L.ref_gstart;
    m.identity_features = L.identity_features;
    m.n_refs = L.n_refs; m.n_features = L.n_features; m.n_words = L.n_words;
    m.n_kmers = L.n_kmers; m.n_classes = L.n_classes; m.n_buckets = L.n_buckets; m.n_spilled = L.n_spilled;
    m.total_gbases = L.total_gbases;
    return m;
}

// ---- index file ---------------------------------------------------------------------------------------------------

static const char kIndexMagic[8] = {'N', 'B', '2', '0', '0', 'I', 'D', 'X'};
static const char *const kSectionName[kIndexSections] = {"feature_names", "tok_end", "tok_comma", "device image"};
constexpr uint64_t kIndexChunk = 64ull << 20;

uint64_t index_checksum(const void *p, uint64_t bytes, uint64_t word0, int threads) {
    const uint8_t *b = static_cast<const uint8_t *>(p);
    const uint64_t nw = bytes / 8;
    std::atomic<uint64_t> sum{0};
    parallel_for(threads, (size_t)nw, [&](int, size_t a, size_t e) {
        uint64_t s = 0;
        for (size_t i = a; i < e; i++) {
            uint64_t w;
            memcpy(&w, b + 8 * i, 8);
            s += image_word_sum(w, word0 + i);
        }
        sum += s;
    });
    uint64_t s = sum;
    if (bytes % 8) {
        uint64_t w = 0;
        memcpy(&w, b + 8 * nw, bytes % 8);
        s += image_word_sum(w, word0 + nw);
    }
    return s;
}

static uint64_t header_checksum(IndexHeader h) {
    h.header_sum = 0;
    return index_checksum(&h, sizeof h, 0);
}

bool is_index_file(const std::string &path) {
    char m[8];
    const int fd = open(path.c_str(), O_RDONLY);
    if (fd < 0) return false;
    const bool yes = pread(fd, m, 8, 0) == 8 && memcmp(m, kIndexMagic, 8) == 0;
    close(fd);
    return yes;
}

static uint64_t align256(uint64_t x) { return (x + 255) & ~(uint64_t)255; }

void write_index_file(const HostLibrary &L, const std::string &json_path, const std::string &out_path, int threads) {
    if (!L.has_index) throw std::runtime_error("library has no k-mer index");
    IndexHeader h{};
    memcpy(h.magic, kIndexMagic, 8);
    h.version = kIndexVersion; h.header_bytes = sizeof(IndexHeader);
    h.sizeof_entry = sizeof(Entry); h.sizeof_classrec = sizeof(ClassRec); h.sizeof_dualrec = sizeof(DualRec);
    const nb200_config &c = L.cfg;
    h.k = (uint32_t)c.k;
    h.score_threshold = c.score_threshold; h.score_filter = c.score_filter; h.num_mismatches = c.num_mismatches;
    h.discard_multiple_matches = c.discard_multiple_matches; h.intersect_level = c.intersect_level;
    h.discard_multi_hits = c.discard_multi_hits; h.require_valid_pair = c.require_valid_pair;
    h.max_hits_to_report = c.max_hits_to_report; h.score_percent = c.score_percent;
    h.n_refs = L.n_refs; h.n_features = L.n_features; h.n_words = L.n_words; h.identity_features = L.identity_features ? 1 : 0;
    h.n_kmers = L.n_kmers; h.n_classes = L.n_classes; h.n_buckets = L.n_buckets; h.n_spilled = L.n_spilled;
    h.total_gbases = L.total_gbases;
    {
        std::ifstream jf(json_path, std::ios::binary);
        if (!jf) throw std::runtime_error("cannot open library file " + json_path);
        uint64_t fnv = 0xCBF29CE484222325ull, n = 0;
        std::vector<char> buf(1 << 20);
        while (jf) {
            jf.read(buf.data(), (std::streamsize)buf.size());
            const std::streamsize got = jf.gcount();
            for (std::streamsize i = 0; i < got; i++) fnv = (fnv ^ (uint8_t)buf[(size_t)i]) * 0x100000001B3ull;
            n += (uint64_t)got;
        }
        h.json_bytes = n; h.json_fnv1a = fnv;
    }
    snprintf(h.lib_version, sizeof h.lib_version, "%s", nb200_version());
    const ImageLayout lay = image_layout(L);
    for (int p = 0; p < kImageParts; p++) h.part_bytes[p] = lay.bytes[p];
    std::string names;
    for (const std::string &s : L.feature_names) { names += s; names.push_back('\0'); }
    const void *host_src[kSecImage] = {names.data(), L.tok_end.data(), L.tok_comma.data()};
    const uint64_t host_bytes[kSecImage] = {names.size(), L.tok_end.size() * 4ull, L.tok_comma.size() * 4ull};
    uint64_t off = align256(sizeof(IndexHeader));
    for (int s = 0; s < kSecImage; s++) {
        h.sec[s] = IndexSection{off, host_bytes[s], index_checksum(host_src[s], host_bytes[s], 0)};
        off = align256(off + host_bytes[s]);
    }
    h.sec[kSecImage] = IndexSection{off, lay.total, 0};
    h.file_bytes = off + lay.total;

    const std::string tmp = out_path + ".tmp";
    FILE *f = fopen(tmp.c_str(), "wb");
    if (!f) throw IoError("cannot write " + tmp);
    try {
        auto put_at = [&](uint64_t at, const void *p, uint64_t n) {
            if (fseeko(f, (off_t)at, SEEK_SET) != 0 || (n && fwrite(p, 1, n, f) != n)) throw IoError("write failed: " + tmp);
        };
        for (int s = 0; s < kSecImage; s++) put_at(h.sec[s].off, host_src[s], host_bytes[s]);
        std::vector<uint8_t> buf(std::min<uint64_t>(kIndexChunk, lay.total));
        uint64_t sum = 0;
        for (uint64_t a = 0; a < lay.total; a += buf.size()) {
            const uint64_t n = std::min<uint64_t>(buf.size(), lay.total - a);
            image_fill(L, lay, a, n, buf.data());
            sum += index_checksum(buf.data(), n, a / 8, threads);
            put_at(h.sec[kSecImage].off + a, buf.data(), n);
        }
        h.sec[kSecImage].sum = sum;
        h.header_sum = header_checksum(h);
        put_at(0, &h, sizeof h);
        const int rc = fclose(f);
        f = nullptr;
        if (rc != 0) throw IoError("write failed: " + tmp);
        if (rename(tmp.c_str(), out_path.c_str()) != 0) throw IoError("cannot rename " + tmp);
    } catch (...) {
        if (f) fclose(f);
        remove(tmp.c_str());
        throw;
    }
}

IndexFile::~IndexFile() { if (fd >= 0) close(fd); }

static void pread_all(int fd, uint64_t at, uint64_t len, uint8_t *dst, const std::string &path) {
    while (len) {
        const ssize_t got = pread(fd, dst, (size_t)std::min<uint64_t>(len, 1ull << 30), (off_t)at);
        if (got < 0 && errno == EINTR) continue;
        if (got <= 0) throw IoError("cannot read index file " + path);
        dst += got; at += (uint64_t)got; len -= (uint64_t)got;
    }
}

void IndexFile::read_image(uint64_t offset, uint64_t len, uint8_t *dst) const {
    pread_all(fd, h.sec[kSecImage].off + offset, len, dst, path);
}

void open_index_file(const std::string &path, IndexFile &f, HostLibrary &meta) {
    auto bad = [&](const std::string &why) { return std::runtime_error("index file " + path + " " + why); };
    f.path = path;
    f.fd = open(path.c_str(), O_RDONLY);
    if (f.fd < 0) throw std::runtime_error("cannot open index file " + path);
    struct stat st;
    if (fstat(f.fd, &st) != 0) throw IoError("cannot stat index file " + path);
    const uint64_t size = (uint64_t)st.st_size;
    if (size < 8) throw bad("is truncated");
    IndexHeader &h = f.h;
    pread_all(f.fd, 0, std::min<uint64_t>(size, sizeof h), reinterpret_cast<uint8_t *>(&h), path);
    if (memcmp(h.magic, kIndexMagic, 8) != 0) throw bad("is not an nb200 index (bad magic)");
    if (size < sizeof h) throw bad("is truncated");
    if (h.version != kIndexVersion)
        throw bad("has format version " + std::to_string(h.version) + "; this build reads version " + std::to_string(kIndexVersion) +
                  " (write it again with `python -m nimble_b200 index`)");
    if (h.header_bytes != sizeof h || h.sizeof_entry != sizeof(Entry) || h.sizeof_classrec != sizeof(ClassRec) ||
        h.sizeof_dualrec != sizeof(DualRec))
        throw bad("was written with a different record layout");
    if (header_checksum(h) != h.header_sum) throw bad("is damaged: the header fails its checksum");
    if (size < h.file_bytes) throw bad("is truncated: " + std::to_string(size) + " of " + std::to_string(h.file_bytes) + " bytes");
    if (size != h.file_bytes) throw bad("has " + std::to_string(size - h.file_bytes) + " bytes after its end");
    const ImageLayout lay = image_layout(h.part_bytes);
    const uint64_t ref_words = (h.total_gbases + 31) / 32 + 2;
    bool ok = h.k >= 4 && h.k <= 32 && h.max_hits_to_report >= 1 && h.max_hits_to_report <= 64 && h.n_refs >= 1 &&
              h.n_refs <= kMaxRefs && h.n_features >= 1 && h.n_features <= h.n_refs && h.n_words == (h.n_refs + 31) / 32 &&
              h.n_buckets >= 1 && h.n_buckets < 0xFFFFFFFFull && h.part_bytes[kPartTable] == h.n_buckets * 2 * sizeof(Entry) &&
              h.part_bytes[kPartClassRec] == h.n_classes * sizeof(ClassRec) && h.part_bytes[kPartRefGstart] == 4ull * h.n_refs &&
              h.part_bytes[kPartRefFeature] == 4ull * h.n_refs && h.part_bytes[kPartRef2bit] == 8 * ref_words &&
              h.part_bytes[kPartRefN] == 4 * ref_words && h.sec[kSecImage].bytes == lay.total &&
              h.sec[kSecTokEnd].bytes == 4ull * h.n_features && h.sec[kSecTokComma].bytes == 4ull * h.n_features;
    for (int s = 0; s < kIndexSections && ok; s++)
        ok = h.sec[s].off % 8 == 0 && h.sec[s].off >= sizeof h && h.sec[s].bytes <= h.file_bytes && h.sec[s].off <= h.file_bytes - h.sec[s].bytes;
    if (!ok) throw bad("is damaged: inconsistent header");
    std::vector<uint8_t> sec[kSecImage];
    for (int s = 0; s < kSecImage; s++) {
        sec[s].resize(h.sec[s].bytes);
        pread_all(f.fd, h.sec[s].off, h.sec[s].bytes, sec[s].data(), path);
        if (index_checksum(sec[s].data(), sec[s].size(), 0) != h.sec[s].sum)
            throw bad(std::string("is damaged: section ") + kSectionName[s] + " fails its checksum");
    }
    meta = HostLibrary{};
    nb200_config &c = meta.cfg;
    c.k = (int32_t)h.k;
    c.score_threshold = h.score_threshold; c.score_filter = h.score_filter; c.num_mismatches = h.num_mismatches;
    c.discard_multiple_matches = h.discard_multiple_matches; c.intersect_level = h.intersect_level;
    c.discard_multi_hits = h.discard_multi_hits; c.require_valid_pair = h.require_valid_pair;
    c.max_hits_to_report = h.max_hits_to_report; c.score_percent = h.score_percent;
    meta.has_index = true;
    const std::vector<uint8_t> &nm = sec[kSecFeatureNames];
    for (size_t a = 0; a < nm.size();) {
        const uint8_t *z = static_cast<const uint8_t *>(memchr(nm.data() + a, 0, nm.size() - a));
        if (!z) throw bad("is damaged: unterminated feature name");
        meta.feature_names.emplace_back(reinterpret_cast<const char *>(nm.data() + a), (size_t)(z - nm.data()) - a);
        a = (size_t)(z - nm.data()) + 1;
    }
    if (meta.feature_names.size() != h.n_features) throw bad("is damaged: feature count differs from the header");
    meta.tok_end.resize(h.n_features); meta.tok_comma.resize(h.n_features);
    memcpy(meta.tok_end.data(), sec[kSecTokEnd].data(), 4ull * h.n_features);
    memcpy(meta.tok_comma.data(), sec[kSecTokComma].data(), 4ull * h.n_features);
    meta.identity_features = h.identity_features != 0;
    meta.n_refs = h.n_refs; meta.n_features = h.n_features; meta.n_words = h.n_words;
    meta.n_kmers = h.n_kmers; meta.n_classes = h.n_classes; meta.n_buckets = h.n_buckets; meta.n_spilled = h.n_spilled;
    meta.total_gbases = h.total_gbases;
}

static bool class_has(const HostLibrary &L, uint32_t c, uint32_t r) {
    if (c >= L.class_rec.size()) return false;
    const ClassRec &rec = L.class_rec[c];
    const uint32_t w = r >> 5, bit = 1u << (r & 31);
    if (rec.meta & kRecOverflow) {
        for (uint64_t j = rec.b[0]; j < (uint64_t)rec.b[0] + rec.b[1] && j < L.ov_w.size() && j < L.ov_b.size(); j++)
            if (L.ov_w[j] == w) return (L.ov_b[j] & bit) != 0;
        return false;
    }
    const uint32_t ws[kRecInline] = {rec.w01 & 0xFFFFu, rec.w01 >> 16, rec.w23 & 0xFFFFu, rec.w23 >> 16};
    for (int i = 0; i < kRecInline; i++)
        if (ws[i] == w) return (rec.b[i] & bit) != 0;
    return false;
}

void verify_index_file(const IndexFile &f, const HostLibrary &meta, int threads) {
    const IndexHeader &h = f.h;
    const ImageLayout lay = image_layout(h.part_bytes);
    uint64_t sum = 0;
    {
        std::vector<uint8_t> buf(std::min<uint64_t>(kIndexChunk, lay.total));
        for (uint64_t a = 0; a < lay.total; a += buf.size()) {
            const uint64_t n = std::min<uint64_t>(buf.size(), lay.total - a);
            f.read_image(a, n, buf.data());
            sum += index_checksum(buf.data(), n, a / 8, threads);
        }
    }
    if (sum != h.sec[kSecImage].sum) throw std::runtime_error("index file " + f.path + " is damaged: the device image fails its checksum");
    HostLibrary L = library_meta(meta);
    auto part = [&](auto &vec, int p) {
        vec.resize(lay.bytes[p] / sizeof(vec[0]));
        f.read_image(lay.off[p], lay.bytes[p], reinterpret_cast<uint8_t *>(vec.data()));
    };
    part(L.table, kPartTable); part(L.class_rec, kPartClassRec); part(L.ov_w, kPartOvW); part(L.ov_b, kPartOvB);
    part(L.ov_pre, kPartOvPre); part(L.positions, kPartPositions); part(L.ref_gstart, kPartRefGstart);
    part(L.ref_feature, kPartRefFeature); part(L.ref2bit, kPartRef2bit); part(L.refN, kPartRefN); part(L.dual, kPartDual);
    // lookup pass: every valid k-mer of every reference, read back from the image, finds a class holding that reference
    const int k = L.cfg.k;
    const uint64_t kmask = k == 32 ? ~0ull : ((1ull << (2 * k)) - 1);
    const uint64_t gend = L.total_gbases >= 128 ? L.total_gbases - 128 : 0;
    std::atomic<uint64_t> bad{0};
    parallel_for(threads, L.n_refs, [&](int, size_t ra, size_t rb) {
        uint64_t nbad = 0;
        for (size_t r = ra; r < rb; r++) {
            const uint64_t g0 = L.ref_gstart[r], g1 = (r + 1 < L.n_refs ? (uint64_t)L.ref_gstart[r + 1] : gend);
            if (g1 < g0 + kRefPad || g1 > gend) { nbad++; continue; }
            uint64_t x = 0;
            int valid = 0;
            for (uint64_t gp = g0; gp < g1 - kRefPad; gp++) {
                if ((L.refN[gp >> 5] >> (gp & 31)) & 1u) { valid = 0; x = 0; continue; }
                const uint64_t c = (L.ref2bit[gp >> 5] >> (2 * (gp & 31))) & 3u;
                x = ((x >> 2) | (c << (2 * (k - 1)))) & kmask;
                if (++valid < k) continue;
                uint32_t cl[2], of[2];
                host_lookup(L, x, cl, of);
                if (cl[0] == kEmptyClass || !class_has(L, cl[0], (uint32_t)r)) nbad++;
            }
        }
        bad += nbad;
    });
    if (bad)
        throw std::runtime_error("index file " + f.path + " is damaged: " + std::to_string((uint64_t)bad) +
                                 " reference k-mers do not find their reference through the table");
}

}  // namespace nb200
