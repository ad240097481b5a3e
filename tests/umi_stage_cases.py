"""Inputs of tests/test_umi_stage_edges_gpu.py, and the host formulas that say where each one sits.

The UMI stage (csrc/agg.cuh, aggregate() and correct_umis() in csrc/engine.cu) picks its code path from the sizes of its
input.  Every case below is built to land on one named side of one of those switches; tests/test_umi_stage_edges.py
recomputes the switch on the host from the same formulas as the engine and fails if a case has moved off its edge.

A case holds CSR rows as nb200_umi_counts takes them (key, off, ids, score) over a library of `names` (byte order).
Cases built from string rows (cell, UMI, comma-joined features, score) keep those rows for the string oracles and the
per-read TSV route; `umis[i]` is row i's UMI string when its key's low half is that UMI's code (or interned id), which
is what lets a case run with UMI correction."""
import itertools
import math

import numpy as np

from nimble_b200.frontend import UMI_CODE_MAX, umi_code, _umi_ids
from oracle import oracle as O
from oracle.a6_py import kahan_sum
from oracle.umi_correct_py import correct_umis

LOCAL_SORT_MAX = 48                 # agg.cuh kLocalSortMax
SMALL_ROWS, SMALL_NAMES = 8, 16     # agg.cuh kSmallRows, kSmallNames
NO_BARCODE = (1 << 64) - 1          # NB200_NO_BARCODE


# ---- the engine's size formulas, restated ------------------------------------------------------------------------
def tok_bits(F):
    """bits of one token column: the smallest b with 2^b >= 2F + 2 (sort_by_feature_string)"""
    b = 1
    while (1 << b) < 2 * F + 2:
        b += 1
    return b


def per_key(F):
    """token columns per 32-bit radix key"""
    return max(1, 32 // tok_bits(F))


def bits_for(n):
    b = 1
    while (1 << b) < n:
        b += 1
    return b


def stage2_bits(D, C):
    """key bits of the stage-2 sort over (cell ordinal, list rank)"""
    return bits_for(D) + bits_for(C) + 1


def slot_table_size(m):
    """slots of the correction table for m selected rows (correct_umis)"""
    t = 1024
    while t < 2 * m and t < (1 << 31):
        t <<= 1
    return t


# ---- cases -------------------------------------------------------------------------------------------------------
class Case:
    def __init__(self, name, names, key, off, ids, score=None, umis=None, rows=None, thresholds=(0.05, 0.3), **claims):
        self.name, self.names = name, names
        self.key = np.ascontiguousarray(key, np.uint64)
        self.off = np.ascontiguousarray(off, np.uint32)
        self.ids = np.ascontiguousarray(ids, np.uint32)
        self.score = None if score is None else np.ascontiguousarray(score, np.float64)
        self.umis, self.rows, self.thresholds, self.claims = umis, rows, thresholds, claims
        self._tok = None

    def __repr__(self):
        return "Case(%s)" % self.name

    @property
    def tok(self):
        if self._tok is None:
            self._tok = O.token_ranks(self.names)
        return self._tok

    def usable(self):
        """rows that reach the UMI stage (mark_rows_kernel)"""
        ok = (self.key != np.uint64(NO_BARCODE)) & (self.off[1:] > self.off[:-1])
        if self.score is not None:
            ok &= ~np.isnan(self.score)
        return ok

    def corrected_key(self):
        """(keys after UMI correction, keys corrected): umi_correct_py.correct_umis on the UMI strings"""
        assert self.umis is not None, self.name
        ok = self.usable()
        rows = [(str(int(k) >> 32) if u else "", self.umis[i], "x" if u else "", 1.0)
                for i, (k, u) in enumerate(zip(self.key.tolist(), ok.tolist()))]
        fixed, n = correct_umis(rows)
        key = self.key.copy()
        ids = umi_ids_map(self.umis)
        for i in np.nonzero(ok)[0]:
            key[i] = (int(self.key[i]) >> 32 << 32) | ids[fixed[i][1]]
        return key, n

    def expected(self, threshold, disable, correct=False):
        """oracle table (cell, count, off, ids, dropped_empty) and the number of keys corrected"""
        key, n = self.corrected_key() if correct else (self.key, 0)
        te, tc = self.tok
        return O.a6_ids(key, self.off.astype(np.int32), self.ids, self.score, te, tc, threshold, disable), n

    def largest_group(self, correct=False):
        key = self.corrected_key()[0] if correct else self.key
        k = key[self.usable()]
        return int(np.unique(k, return_counts=True)[1].max()) if len(k) else 0

    def selected(self):
        return int(self.usable().sum())

    def max_nf(self):
        ok = self.usable()
        return int((self.off[1:] - self.off[:-1])[ok].max())


def umi_ids_map(umis):
    u = sorted(set(umis))
    return dict(zip(u, (int(x) for x in _umi_ids(u))))


def from_rows(name, rows, extra_names=(), **kw):
    """string rows (cell, UMI, comma-joined features, score) -> Case, keyed as `report` keys them: cells by byte order,
    the UMI's code (frontend.umi_code) or its interned id"""
    names = sorted({x for r in rows if r[2] for x in r[2].split(",")} | set(extra_names))
    fid = {n: i for i, n in enumerate(names)}
    cbs = sorted({r[0] for r in rows})
    cid = {c: i for i, c in enumerate(cbs)}
    umap = umi_ids_map([r[1] for r in rows])
    key = np.array([(cid[r[0]] << 32) | umap[r[1]] for r in rows], np.uint64)
    off = np.zeros(len(rows) + 1, np.uint32)
    ids = []
    for i, r in enumerate(rows):
        ids.extend(sorted(fid[x] for x in r[2].split(",")) if r[2] else [])
        off[i + 1] = len(ids)
    c = Case(name, names, key, off, np.array(ids, np.uint32), [float(r[3]) for r in rows], [r[1] for r in rows], list(rows), **kw)
    c.cbs = cbs
    return c


def csr(lists):
    off = np.zeros(len(lists) + 1, np.uint32)
    np.cumsum([len(l) for l in lists], out=off[1:])
    return off, np.array([x for l in lists for x in l], np.uint32)


def random_umis(rng, n, length=10):
    """n distinct ACGT UMIs of one length"""
    out, seen = [], set()
    while len(out) < n:
        for row in rng.integers(0, 4, size=(n, length)):
            u = "".join("ACGT"[x] for x in row)
            if u not in seen:
                seen.add(u)
                out.append(u)
                if len(out) == n:
                    break
    return out


def mutate(rng, umi):
    p = int(rng.integers(0, len(umi)))
    return umi[:p] + str(rng.choice([c for c in "ACGT" if c != umi[p]])) + umi[p + 1:]


# ---- 1. token packing --------------------------------------------------------------------------------------------
HLA = ["A", "A*01", "A*01:01", "A+B", "A-1", "A 2"]      # byte order differs from comma-joined order: ' ' '+' < ','


def hla_names(F):
    """F names in byte order: the HLA-style set, then stems with the same six suffixes (shared prefixes, bytes below ',')"""
    out = list(HLA[:F])
    i = 0
    while len(out) < F:
        s, j = "", i // 6
        while True:
            s = "0123456789BCDFGHJKLMPQRSVWXZ"[j % 28] + s
            j //= 28
            if not j:
                break
        out.append("H" + s + ["", "*01", "*01:01", "+B", "-1", " 2"][i % 6])
        i += 1
    return sorted(out, key=str.encode)


def token_max_nf(F):
    """longest row per residue of max_nf modulo per_key: 0, 1 and per_key - 1, each at least 3 per_key + 1"""
    pk = per_key(F)
    lo = 3 * pk + 1
    return sorted({lo + (r - lo) % pk for r in (0, 1 % pk, pk - 1)})


def token_case(F, max_nf, big, seed=0, names=None):
    """rows of 1..max_nf names over F features (shared prefixes, the highest and lowest ids, identical lists within a
    UMI); every group <= 48 rows, or (big) one group of 49"""
    rng = np.random.default_rng([F, max_nf, int(big), seed])
    names = names or hla_names(F)
    lists, key, umis = [], [], []
    hi = [F - 1 - x for x in range(min(F, 8))]
    pools = []
    for c in range(6):
        base = rng.choice(F, size=max_nf * 2, replace=False).tolist()
        base[0] = hi[c % len(hi)]
        pools.append(base)
    n_umis = 240
    umi_strs = random_umis(rng, n_umis + 1, 8)
    for g in range(n_umis + 1):
        cell = g % 6
        rows = LOCAL_SORT_MAX + 1 if (big and g == n_umis) else (int(rng.integers(1, 6)) if g < n_umis else 0)
        pool = pools[cell]
        mine = []
        for r in range(rows):
            if mine and rng.random() < 0.3:
                l = mine[int(rng.integers(0, len(mine)))]              # an identical list, later in input order
            else:
                L = max_nf if (g + r) % 7 == 0 else int(rng.integers(1, max_nf + 1))
                if rng.random() < 0.6:
                    l = sorted(pool[:L - 1] + [int(rng.integers(0, F))])   # shared prefix, differs late
                else:
                    l = sorted(int(x) for x in rng.choice(F, size=L, replace=False))
            mine.append(l)
            lists.append(l)
            key.append((cell << 32) | umi_code(umi_strs[g]))
            umis.append(umi_strs[g])
    lists.append(sorted(pool[:max_nf]))                                # at least one row of max_nf names
    key.append((5 << 32) | umi_code(umi_strs[0]))
    umis.append(umi_strs[0])
    perm = rng.permutation(len(lists))                                 # rows of a UMI interleave with other UMIs
    lists = [lists[i] for i in perm]
    off, ids = csr(lists)
    return Case("token_F%d_nf%d_%s" % (F, max_nf, "g49" if big else "g48"), names, np.array(key, np.uint64)[perm], off, ids,
                None, [umis[i] for i in perm], F=F, max_nf=max_nf, big=big)


# ---- 2. group sort and 7. float edges: order-sensitive Kahan sums ---------------------------------------------------
# Kahan sum of these four scores in this order is below their Kahan sum in every other order (a stable-sort bug
# reorders them), and t / (sum + t) moves with it.
KAHAN_SET = [362.88354522312784, 9.44876581664646, 88.98328784288333, 0.8566941897809504]


def kahan_threshold(values=KAHAN_SET):
    """(t, threshold): the ratio of a one-row feature of score t beside a merged row of `values` is exactly the
    threshold in input order, and below it in any other order"""
    f = kahan_sum(values)
    t = f * 0.1
    return t, t / (f + t)


def kahan_rows(n_rows, cell="CELL0", umi="GRP"):
    """one UMI of n_rows rows in reverse feature-string order: "B" (score t) first, then the four KAHAN_SET rows of list
    "A" interleaved with zero-score "A,C" rows.  At the threshold B is kept and the UMI's intersection is empty; with
    the four "A" rows summed in any other order, B falls below it and the UMI counts "A"."""
    t, _ = kahan_threshold()
    out = [(cell, umi, "B", t)]
    at = [1 + j * ((n_rows - 2) // len(KAHAN_SET)) for j in range(len(KAHAN_SET))]
    for i in range(n_rows - 1):
        out.append((cell, umi, "A", KAHAN_SET[at.index(i)]) if i in at else (cell, umi, "A,C", 0.0))
    return out


def group_sort_case(n):
    _, thr = kahan_threshold()
    rows = kahan_rows(n)
    rows += [("CELL1", "U%02d" % i, ["A", "B", "A,B", "C"][i % 4], 1.0 + i) for i in range(12)]
    return from_rows("group_sort_%d" % n, rows, thresholds=(thr, math.nextafter(thr, 1.0), 0.05), largest=n)


# ---- 3. general-kernel working set -------------------------------------------------------------------------------
def general_rows(n_rows, n_names, umi):
    """one UMI of n_rows rows and n_names names in all, not one list: every row holds "S"; row j holds "x<j>_<t>" too"""
    base, extra = divmod(n_names, n_rows)
    out = []
    for j in range(n_rows):
        L = base + (1 if j < extra else 0)
        out.append(("CELLG", umi, ",".join(["S"] + ["x%d_%d" % (j, t) for t in range(L - 1)]), 1.0 + 0.25 * j))
    return out


def general_case():
    rows, shapes = [], [(8, 16), (9, 16), (8, 17), (9, 17)]
    for r, n in shapes:
        rows += general_rows(r, n, "W%d_%d" % (r, n))
    # one list with a duplicated name: the general kernel, small and not
    rows += [("CELLG", "D8", "D,D", 1.0)] * 8 + [("CELLG", "D9", "D,D", 1.0)] * 9
    rows += [("CELLG", "D1", ",".join(["E"] * 3 + ["E%02d" % i for i in range(14)]), 2.0)]
    rows += [("CELLH", "P%d" % i, "S", 1.0) for i in range(5)]
    shapes += [(8, 16), (9, 18), (1, 17)]
    return from_rows("general", rows, general={u: s for u, s in zip(["W8_16", "W9_16", "W8_17", "W9_17", "D8", "D9", "D1"], shapes)})


# ---- 4. stage-2 key width ----------------------------------------------------------------------------------------
def stage2_case(C, D, seed=0, thresholds=(0.3,)):
    """G = max(C, D) UMIs of one row each (simple kernel, ratios >= 1/2: every list survives); UMI g is in cell g % C
    and carries distinct list g % D, both through random permutations.  Three more UMIs hold two rows with disjoint
    lists each: they end without a result, so the stage-2 sort also carries its sentinel key (bit rank_bits + cell_bits,
    the top bit of the sort)."""
    rng = np.random.default_rng([C, D, seed])
    F = 2
    while F + F * (F - 1) // 2 < D:
        F += 1
    names = ["f%05d" % i for i in range(F)]
    all_lists = [[i] for i in range(F)] + [[i, j] for i in range(F) for j in range(i + 1, F)]
    pick = rng.permutation(len(all_lists))[:D]
    G = max(C, D)
    g = np.arange(G)
    cell = rng.permutation(C)[g % C].astype(np.uint64)
    flat = [all_lists[pick[x]] for x in rng.permutation(D)]
    other = next(l for l in flat if len(l) == len(flat[0]) and set(l).isdisjoint(flat[0]))    # no result at any threshold
    perm = rng.permutation(G)
    extra_cell = cell[:3].repeat(2)
    extra_lists = [flat[0], other] * 3
    if G <= 200_000:                 # UMI strings (correction can run)
        umis = random_umis(rng, G + 3, 12)
        umis = [umis[i] for i in perm] + [u for u in umis[G:] for _ in range(2)]
        key = np.concatenate([cell[perm], extra_cell]) << np.uint64(32) | np.array([umi_code(u) for u in umis], np.uint64)
        off, ids = csr([flat[x] for x in (g % D)[perm]] + extra_lists)
        return Case("stage2_C%d_D%d" % (C, D), names, key, off, ids, None, umis, thresholds=thresholds, C=C, D=D)
    # a million UMIs: keys and CSR straight from numpy (UMI g's low half is g + 1, a code)
    key = np.concatenate([(cell[perm] << np.uint64(32)) | (perm + 1).astype(np.uint64),
                          (extra_cell << np.uint64(32)) | np.arange(G + 1, G + 4, dtype=np.uint64).repeat(2)])
    a = np.array([l[0] for l in flat], np.uint32)
    b = np.array([l[-1] for l in flat], np.uint32)
    two = np.array([len(l) == 2 for l in flat])
    d = (g % D)[perm]
    off = np.zeros(G + 1, np.uint32)
    np.cumsum(np.where(two[d], 2, 1), out=off[1:])
    ids = np.empty(int(off[-1]), np.uint32)
    ids[off[:-1]] = a[d]
    ids[off[:-1][two[d]] + 1] = b[d][two[d]]
    eo, ei = csr(extra_lists)
    off = np.concatenate([off, off[-1] + eo[1:]])
    ids = np.concatenate([ids, ei])
    return Case("stage2_C%d_D%d" % (C, D), names, key, off, ids, None, None, thresholds=thresholds, C=C, D=D)


# ---- 5. count width and cells ------------------------------------------------------------------------------------
def count_width_case():
    """cell 7: lists "c255", "c256", "c70000" with that many UMIs each; cell 9: 66 000 distinct lists, one UMI each"""
    rng = np.random.default_rng(5)
    P = 400
    names = ["c255", "c256", "c70000"] + ["p%03d" % i for i in range(P)]
    names.sort()
    fid = {n: i for i, n in enumerate(names)}
    lists, cells = [], []
    for n, c in (("c255", 255), ("c256", 256), ("c70000", 70000)):
        lists += [[fid[n]]] * c
        cells += [7] * c
    pairs = [[fid["p%03d" % i], fid["p%03d" % j]] for i in range(P) for j in range(i + 1, P)]
    pick = rng.permutation(len(pairs))[:66000]
    lists += [pairs[i] for i in pick]
    cells += [9] * len(pick)
    umis = random_umis(rng, len(lists), 12)
    key = (np.array(cells, np.uint64) << np.uint64(32)) | np.array([umi_code(u) for u in umis], np.uint64)
    perm = rng.permutation(len(lists))
    off, ids = csr([lists[i] for i in perm])
    return Case("count_width", names, key[perm], off, ids, None, [umis[i] for i in perm], counts=(255, 256, 70000),
                cell_rows=66000)


# ---- 6. keys -----------------------------------------------------------------------------------------------------
def keys_case():
    """cell halves with bit 31 set and 0xFFFFFFFF (legal; only NB200_NO_BARCODE is dropped), keys one bit apart at
    bits 0, 32 and 63, each with its own list; NB200_NO_BARCODE rows that must not count"""
    names = ["k%d" % i for i in range(10)]
    spec = [
        (0xFFFFFFFF, 0xFFFFFFFE, [0]), (0xFFFFFFFF, 0, [1]), (0xFFFFFFFF, 7, [0, 1]),
        (0x80000000, 3, [2]), (0x80000001, 3, [2]), (0xFFFFFFFE, 9, [3]),
        (0x10, 2, [4]), (0x10, 3, [5]),                      # bit 0
        (0x20, 5, [6]), (0x21, 5, [6]),                      # bit 32
        (0x30, 5, [7]), (0x80000030, 5, [8]),                # bit 63
        (0x30, 6, [7]), (0x30, 6, [9]),                      # one UMI, two lists: empty intersection
    ]
    key = [(c << 32) | u for c, u, _ in spec] + [NO_BARCODE] * 3
    lists = [l for _, _, l in spec] + [[0], [1], [2]]
    key += key[:6]
    lists += lists[:6]
    off, ids = csr(lists)
    return Case("keys", names, np.array(key, np.uint64), off, ids, None)


def many_keys_case(n=4_200_000):
    """n distinct keys of one row each: 5 000 cells x random 32-bit UMIs; lists from 24 single names"""
    rng = np.random.default_rng(6)
    key = np.sort((rng.integers(0, 5000, size=int(n * 1.01)).astype(np.uint64) << np.uint64(32))
                  | rng.integers(0, 1 << 32, size=int(n * 1.01), dtype=np.uint64))
    key = rng.permutation(key[np.concatenate([[True], key[1:] != key[:-1]])])[:n]
    names = ["m%02d" % i for i in range(24)]
    off = np.arange(n + 1, dtype=np.uint32)
    ids = rng.integers(0, 24, size=n).astype(np.uint32)
    return Case("many_keys", names, key, off, ids, None, thresholds=(0.05,))


# ---- 7. float edges ----------------------------------------------------------------------------------------------
def float_edges_case():
    inf, nan = float("inf"), float("nan")
    rows = [
        ("C1", "Z0", "A", 0.0), ("C1", "Z0", "B", 0.0),               # total zero: 0/0 ratios are kept
        ("C1", "Z1", "A,B", 0.0),
        ("C1", "I0", "A", inf), ("C1", "I0", "B", 1.0),               # 1/inf = 0 < threshold
        ("C1", "I1", "A", inf), ("C1", "I1", "A", -inf),              # merged row of nan
        ("C1", "I2", "A,B", inf),
        ("C2", "M0", "A", -0.0), ("C2", "M0", "A,B", -0.0),
        ("C2", "N0", "A", nan),                                       # NaN rows do not count
        ("C2", "N1", "A", nan), ("C2", "N1", "B", 1.0),
        ("C2", "N2", "A,B", nan), ("C2", "N2", "A,B", 1.0), ("C2", "N2", "A", 3.0),
    ]
    return from_rows("float_edges", rows)


def knife_simple_case():
    """a one-list UMI of three names: ratio (1/3)/1; at that threshold kept, one ulp above it dropped"""
    thr = (1.0 / 3.0) / 1.0
    rows = [("C3", "K0", "A,B,C", 1.0), ("C3", "K1", "D", 1.0)]
    return from_rows("knife_simple", rows, thresholds=(thr, math.nextafter(thr, 1.0)))


def knife_general_case():
    """B's ratio 0.1 / (0.7 + 0.1) as the general kernel computes it: kept at that threshold, dropped one ulp above"""
    thr = 0.1 / (0.7 + 0.1)
    rows = [("C3", "K2", "A", 0.7), ("C3", "K2", "B", 0.1), ("C3", "K3", "D", 1.0)]
    return from_rows("knife_general", rows, thresholds=(thr, math.nextafter(thr, 1.0)))


def kahan_small_case():
    """the Kahan set on merged rows of a six-row UMI (thread-local working set)"""
    _, thr = kahan_threshold()
    return from_rows("kahan_small", kahan_rows(6), thresholds=(thr, math.nextafter(thr, 1.0)))


# ---- 8. correction -----------------------------------------------------------------------------------------------
def grow_past_48_case():
    """40 rows of one UMI and 9 of its neighbour: every group <= 48 without correction, 49 with it"""
    rng = np.random.default_rng(8)
    u, v = "ACGTACGTACGT", "ACGTACGAACGT"
    rows = [("CELLA", u, ["f1", "f1,f2", "f2,f3"][i % 3], 1.0 + (i % 5) * 0.5) for i in range(40)]
    rows += [("CELLA", v, "f1,f2", 0.75) for _ in range(9)]
    rows += [("CELLC", mutate(rng, u), "f1", 1.0) for _ in range(8)]
    rows += [("CELLC", u, "f1", 1.0) for _ in range(20)]
    order = rng.permutation(len(rows))
    return from_rows("grow_past_48", [rows[i] for i in order], largest=(40, 49))


def big_umi_case():
    """a 2 500-row UMI with 30 one-row neighbours"""
    rng = np.random.default_rng(9)
    w = "TTGCAAGCTTGA"
    rows = [("CELLB", w, ["g1", "g1,g2", "g1,g3"][i % 3], 1.0) for i in range(2500)]
    nb = set()
    while len(nb) < 30:
        nb.add(mutate(rng, w))
    rows += [("CELLB", x, "g1,g%d" % (2 + i % 3), 1.0) for i, x in enumerate(sorted(nb))]
    order = rng.permutation(len(rows))
    return from_rows("big_umi", [rows[i] for i in order], largest=(2500, 2530))


def one_base_case():
    rows = []
    for cell, counts in (("C1", dict(A=3, C=3, G=2, T=1, N=1)), ("C2", dict(N=5, A=1)), ("C3", dict(G=2, T=2, N=2, A=1, C=1))):
        for b, n in counts.items():
            rows += [(cell, b, ["F", "F,G", "H"][i % 3], 1.0) for i in range(n)]
    return from_rows("one_base", rows)


def thirteen_case():
    """13-base UMIs at the top of the code: N x13 (= UMI_CODE_MAX), T x13, an N at each position; other lengths and
    interned UMIs in the same cell"""
    assert umi_code("N" * 13) == UMI_CODE_MAX
    rows = [("C1", "N" * 13, "F", 1.0), ("C1", "N" * 12 + "A", "F", 1.0), ("C1", "N" * 12 + "A", "F,G", 1.0)]
    rows += [("C1", "T" * 13, "G", 1.0)] * 3 + [("C1", "T" * 12 + "G", "G", 1.0)]
    rows += [("C1", "A" * 13, "H", 1.0)] * 4
    rows += [("C1", "A" * p + "N" + "A" * (12 - p), ["H", "H,F"][p % 2], 1.0) for p in range(13)]
    rows += [("C1", "A" * 12, "H", 1.0), ("C1", "A" * 12, "H", 1.0), ("C1", "A" * 11 + "C", "H", 1.0),
             ("C1", "A" * 14, "H", 1.0), ("C1", "A" * 13 + "C", "H", 1.0), ("C1", "ACGX", "F", 1.0), ("C1", "A", "F", 1.0)]
    rows += [("C2", "N" * 13, "F", 1.0)] * 2 + [("C2", "N" * 6 + "C" + "N" * 6, "F", 1.0)]
    return from_rows("thirteen", rows)


def selected_rows_case(m, seed=0):
    """exactly m rows that count (10-base UMIs in 16 cells, 5 % one substitution from another row's UMI), and rows that
    must not move m: NaN score, empty list, NB200_NO_BARCODE"""
    rng = np.random.default_rng([m, seed])
    base = random_umis(rng, m, 10)
    rows = []
    for i in range(m):
        cell = "CELL%02d" % rng.integers(0, 16)
        umi = base[i]
        if i and rng.random() < 0.05:
            j = int(rng.integers(0, len(rows)))
            cell, umi = rows[j][0], mutate(rng, rows[j][1])
        rows.append((cell, umi, "f%d" % rng.integers(0, 6), 1.0))
    rows += [("CELL00", base[0], "f1", float("nan")), ("CELL01", base[1], "", 1.0), ("CELL02", mutate(rng, base[2]), "", 2.0)]
    c = from_rows("m%d" % m, rows, thresholds=(0.05,), m=m)
    c.rows = None                                  # NB200_NO_BARCODE rows exist only as keys
    c.key = np.concatenate([c.key, np.full(3, NO_BARCODE, np.uint64)])
    c.off = np.concatenate([c.off, c.off[-1] + np.array([1, 2, 3], np.uint32)])
    c.ids = np.concatenate([c.ids, np.zeros(3, np.uint32)])
    c.score = np.concatenate([c.score, np.ones(3)])
    c.umis = c.umis + [base[0]] * 3
    return c


SELECTED_M = [511, 512, 513, (1 << 15) - 1, 1 << 15, (1 << 15) + 1]


def ties_case():
    """a one-row UMI with 18 three-row neighbours: the byte order of the UMIs decides every target"""
    x = "CCCCCC"
    rows = [("C1", x, "F", 1.0)]
    for p in range(6):
        for b in "AGT":
            rows += [("C1", x[:p] + b + x[p + 1:], ["F", "F,G"][p % 2], 1.0)] * 3
    rows += [("C2", "ACGT", "F", 1.0)] * 2 + [("C2", "ACGA", "F", 1.0)] * 2 + [("C2", "ACGC", "F", 1.0)] * 2 + [("C2", "ACGG", "F", 1.0)]
    return from_rows("ties", rows)


# ---- 10. seeded sweep ---------------------------------------------------------------------------------------------
def sweep_case(seed):
    """one case within +-2 of a switch, drawn from the seed"""
    rng = np.random.default_rng(seed)
    kind = ["token", "group", "general", "stage2"][seed % 4]
    if kind == "token":
        F = int(rng.choice([127, 128, 511, 512, 32767, 32768])) + int(rng.integers(-2, 3))
        pk = per_key(F)
        c = token_case(F, 3 * pk + 1 + int(rng.integers(-2, 3)), bool(rng.integers(0, 2)), seed)
    elif kind == "group":
        n = LOCAL_SORT_MAX + int(rng.integers(-2, 3))
        rows = [("CELL0", "ACGTAC", ["A", "A,B", "B", "A,C"][int(rng.integers(0, 4))], float(rng.choice([0.5, 1.0, 2.0, 0.1])))
                for i in range(n)]
        rows += [("CELL0", mutate(rng, "ACGTAC"), ["A", "B"][i % 2], 1.0) for i in range(int(rng.integers(0, 5)))]
        rows += [("CELL%d" % (1 + i % 2), random_umis(rng, 1, 6)[0], "A", 1.0) for i in range(10)]
        rows = [rows[i] for i in rng.permutation(len(rows))]
        c = from_rows("sweep_group", rows)
    elif kind == "general":
        rows = []
        for g in range(6):
            r = SMALL_ROWS + int(rng.integers(-2, 3))
            n = max(r, SMALL_NAMES + int(rng.integers(-2, 3)))
            rows += general_rows(r, n, random_umis(rng, 1, 8)[0] + "AC"[g % 2])
        c = from_rows("sweep_general", rows)
    else:
        k = int(rng.integers(9, 14))
        C = (1 << int(rng.integers(4, 9))) + int(rng.integers(-2, 3))
        c = stage2_case(C, (1 << k) + int(rng.integers(-2, 3)), seed, thresholds=(0.05,))
    c.name = "sweep%d_%s" % (seed, c.name)
    c.claims["kind"] = kind
    return c


def permutations_differ(values=KAHAN_SET):
    """every other order of `values` has a larger Kahan sum, and moves the ratio of kahan_threshold below it"""
    t, thr = kahan_threshold(values)
    f = kahan_sum(values)
    for p in itertools.permutations(values):
        if list(p) == list(values):
            continue
        o = kahan_sum(list(p))
        if not (o > f and t / (o + t) < thr):
            return False
    return True
