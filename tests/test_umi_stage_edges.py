"""The inputs of tests/test_umi_stage_edges_gpu.py sit where they claim (no GPU).

Each case is built to land on one side of a size switch of the UMI stage.  Here the switch is recomputed on the host
from the engine's own formulas, so that an edit to a generator cannot move a case off its edge unnoticed; the
order-sensitive scores and the knife-edge thresholds are shown to change the oracle's output; and the C oracle the GPU
file compares with agrees with the string oracle wherever both can run."""
import math
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import umi_stage_cases as U
from oracle import a6_py
from oracle.a6_py import report_counts
from oracle.umi_correct_py import correct_umis

TOKEN_F = [127, 128, 511, 512, 32767, 32768, 200_000]


def strings(case, table):
    """C oracle table -> [(features, count, cell string)] as report_counts gives it"""
    cell, cnt, off, ids, dropped = table
    return [(",".join(case.names[j] for j in ids[off[i]:off[i + 1]]), int(cnt[i]), case.cbs[cell[i]]) for i in range(len(cell))], dropped


def test_engine_formulas():
    assert [(U.tok_bits(F), U.per_key(F)) for F in TOKEN_F] == [(8, 4), (9, 3), (10, 3), (11, 2), (16, 2), (17, 1), (19, 1)]
    assert [U.slot_table_size(m) for m in U.SELECTED_M] == [1024, 1024, 2048, 65536, 65536, 131072]
    assert U.bits_for(1) == 1 and U.bits_for(1 << 16) == 16 and U.bits_for((1 << 16) + 1) == 17


@pytest.mark.parametrize("F", TOKEN_F)
def test_token_cases_sit_on_their_switch(F):
    pk = U.per_key(F)
    nfs = U.token_max_nf(F)
    assert {nf % pk for nf in nfs} == {0, 1 % pk, pk - 1}
    names = U.hla_names(F)
    assert len(set(names)) == F and names == sorted(names, key=str.encode)
    if F >= len(U.HLA):
        assert set(U.HLA) <= set(names)
    for nf in nfs:
        assert nf >= 3 * pk + 1
        for big in (False, True):
            c = U.token_case(F, nf, big, names=names)
            assert c.max_nf() == nf
            assert np.all(c.ids < F) and int(c.ids.max()) >= F - 8     # the top token ranks are in use
            g = c.largest_group()
            assert (g == U.LOCAL_SORT_MAX + 1) if big else (g <= U.LOCAL_SORT_MAX)


def test_hla_byte_order_differs_from_string_order():
    c = U.token_case(127, 16, False)
    te, tc = c.tok
    i = {n: k for k, n in enumerate(c.names)}
    # "A" < "A 2" by id, but "A 2" < "A,<any>" as comma-joined strings
    assert i["A"] < i["A 2"] and te[i["A 2"]] < tc[i["A"]]
    assert i["A"] < i["A+B"] and te[i["A+B"]] < tc[i["A"]]


@pytest.mark.parametrize("n", [48, 49])
def test_group_sort_cases(n):
    c = U.group_sort_case(n)
    assert c.largest_group() == n == c.claims["largest"]
    grp = [r[2] for r in c.rows if r[1] == "GRP"]
    assert grp[0] == "B" and grp != sorted(grp)                        # not in feature-string order
    assert sum(1 for a, b in zip(grp, grp[1:]) if a != b) >= 6         # identical lists apart from each other


def test_kahan_set_is_order_sensitive():
    assert U.permutations_differ()
    _, thr = U.kahan_threshold()
    for rows in (U.kahan_rows(48), U.kahan_rows(6)):
        want = report_counts(rows, thr)
        assert want == ([], 1)                                          # B kept: the intersection is empty
        a = [i for i, r in enumerate(rows) if r[2] == "A"]
        for perm in ([3, 2, 1, 0], [1, 0, 2, 3], [0, 1, 3, 2]):       # the "A" rows in another order
            moved = list(rows)
            for i, p in zip(a, perm):
                moved[i] = rows[a[p]]
            assert report_counts(moved, thr) == ([("A", 1, "CELL0")], 0)


def test_kahan_sum_matters_here():
    """a plain left-to-right sum of the same rows gives another table: the sets test the compensation itself"""
    _, thr = U.kahan_threshold()
    rows = U.kahan_rows(48)
    saved = a6_py.kahan_sum

    def plain(v):
        s = 0.0
        for x in v:
            s += x
        return s
    a6_py.kahan_sum = plain
    try:
        got = report_counts(rows, thr)
    finally:
        a6_py.kahan_sum = saved
    assert got != report_counts(rows, thr)


@pytest.mark.parametrize("make", [U.knife_simple_case, U.knife_general_case, U.kahan_small_case, lambda: U.group_sort_case(48)])
def test_knife_edges_are_knife_edges(make):
    c = make()
    thr = c.thresholds[0]
    at, _ = c.expected(thr, False)
    above, _ = c.expected(math.nextafter(thr, 1.0), False)
    below, _ = c.expected(math.nextafter(thr, 0.0), False)
    assert strings(c, at) != strings(c, above)
    assert strings(c, at) == strings(c, below)
    assert report_counts(c.rows, thr) == strings(c, at)
    assert report_counts(c.rows, math.nextafter(thr, 1.0)) == strings(c, above)


def test_general_cases():
    c = U.general_case()
    for umi, (nr, nn) in c.claims["general"].items():
        rows = [r for r in c.rows if r[1] == umi]
        lists = [r[2].split(",") for r in rows]
        assert len(rows) == nr and sum(len(l) for l in lists) == nn, umi
        assert len({r[2] for r in rows}) > 1 or any(len(set(l)) < len(l) for l in lists), umi    # general kernel
    small = {u for u, (nr, nn) in c.claims["general"].items() if nr <= U.SMALL_ROWS and nn <= U.SMALL_NAMES}
    assert small == {"W8_16", "D8"}


def _list_codes(c):
    first = c.ids[c.off[:-1]].astype(np.int64)
    two = (c.off[1:] - c.off[:-1]) == 2
    second = np.where(two, c.ids[np.minimum(c.off[:-1] + 1, len(c.ids) - 1)], len(c.names)).astype(np.int64)
    return first * (len(c.names) + 1) + second


STAGE2 = [((1 << 15), (1 << 16), 32), ((1 << 15), (1 << 16) + 1, 33), ((1 << 20) + 1, (1 << 17) + 1, 40),
          (1, 1 << 16, None), (1, (1 << 16) + 1, None)]


@pytest.mark.parametrize("C,D,bits", STAGE2)
def test_stage2_cases(C, D, bits):
    if bits is not None:
        assert U.stage2_bits(D, C) == bits
    c = U.stage2_case(C, D)
    assert len(np.unique(c.key >> np.uint64(32))) == C
    assert len(np.unique(_list_codes(c))) == D                      # one row per UMI, every list survives
    assert np.all((c.off[1:] - c.off[:-1]) <= 2)
    k = np.sort(c.key)
    assert int((k[1:] == k[:-1]).sum()) == 3 and len(c.key) == max(C, D) + 6


def test_stage2_sentinel():
    """three UMIs of every stage-2 case end without a result: the sort's top key bit is in use"""
    for C, D in ((5, 300), (1 << 15, (1 << 16) + 1)):
        c = U.stage2_case(C, D)
        full = c.expected(0.3, False)[0]
        assert c.expected(0.3, True)[0][4] == 3
        n = max(C, D)                                   # the same table without the three UMIs
        c.key, c.off, c.ids, c.umis = c.key[:n], c.off[:n + 1], c.ids[:int(c.off[n])], None
        assert all(np.array_equal(a, b) for a, b in zip(full[:4], c.expected(0.3, False)[0][:4]))


def test_stage2_small_case_through_the_oracle():
    c = U.stage2_case(3, 1000)
    (cell, cnt, off, ids, dropped), _ = c.expected(0.3, False)
    assert len({tuple(ids[off[i]:off[i + 1]]) for i in range(len(cell))}) == 1000 and len(set(cell.tolist())) == 3


def test_count_width_case():
    c = U.count_width_case()
    (cell, cnt, off, ids, dropped), _ = c.expected(0.05, False)
    assert set(cnt[cell == 7].tolist()) == {255, 256, 70000}
    assert int((cell == 9).sum()) == 66000 > 65536


def test_keys_case():
    c = U.keys_case()
    k = c.key.tolist()
    assert k.count(U.NO_BARCODE) == 3
    assert any(x >> 32 == 0xFFFFFFFF and x != U.NO_BARCODE for x in k)
    assert any(x >> 63 for x in k if x != U.NO_BARCODE)
    for bit in (0, 32, 63):
        assert any((x ^ (1 << bit)) in k for x in k if x != U.NO_BARCODE), bit
    (cell, cnt, off, ids, dropped), _ = c.expected(0.05, False)
    assert 0xFFFFFFFF in cell.tolist() and dropped == 1


def test_many_keys_case():
    c = U.many_keys_case()
    k = np.sort(c.key)
    assert len(k) >= 4_000_000 and np.all(k[1:] != k[:-1])
    x = c.key.copy()                                 # a 32-bit hash of the key (murmur3 fmix64, low half)
    x ^= x >> np.uint64(33); x *= np.uint64(0xFF51AFD7ED558CCD); x ^= x >> np.uint64(33)
    x *= np.uint64(0xC4CEB9FE1A85EC53); x ^= x >> np.uint64(33)
    h = (x & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    h.sort()
    assert int((h[1:] == h[:-1]).sum()) > 1000


def test_one_base_thirteen_and_ties():
    one = U.one_base_case()
    assert {r[1] for r in one.rows if r[0] == "C1"} == set("ACGTN")
    t = U.thirteen_case()
    umis = {r[1] for r in t.rows if r[0] == "C1"}
    assert {"N" * 13, "T" * 13} <= umis and all("A" * p + "N" + "A" * (12 - p) in umis for p in range(13))
    assert {len(u) for u in umis} >= {1, 4, 12, 13, 14} and "ACGX" in umis
    fixed, n = correct_umis(U.ties_case().rows)
    # the one-row UMI has 18 neighbours of three rows: the byte order alone picks TCCCCC; each neighbour moves to the
    # T at its own position
    assert fixed[0][1] == "TCCCCC" and all("T" in r[1] for r in fixed if r[0] == "C1") and n >= 13


@pytest.mark.parametrize("make", [U.grow_past_48_case, U.big_umi_case])
def test_correction_grows_groups(make):
    c = make()
    before, after = c.claims["largest"]
    assert c.largest_group() == before and c.largest_group(correct=True) == after
    if make is U.grow_past_48_case:
        assert before <= U.LOCAL_SORT_MAX < after


@pytest.mark.parametrize("m", U.SELECTED_M)
def test_selected_rows_cases(m):
    c = U.selected_rows_case(m)
    assert c.selected() == m and len(c.key) == m + 6
    assert c.corrected_key()[1] > 0


SMALL = [U.float_edges_case, U.knife_simple_case, U.knife_general_case, U.kahan_small_case, lambda: U.group_sort_case(48),
         lambda: U.group_sort_case(49), U.general_case, U.one_base_case, U.thirteen_case, U.ties_case, U.grow_past_48_case]


@pytest.mark.parametrize("k", range(len(SMALL)))
def test_c_oracle_equals_string_oracle(k):
    c = SMALL[k]()
    for thr in tuple(c.thresholds) + (0.05,):
        for dis in (False, True):
            assert strings(c, c.expected(thr, dis)[0]) == report_counts(c.rows, thr, dis), (c.name, thr, dis)
            fixed, n = correct_umis(c.rows)
            table, n2 = c.expected(thr, dis, True)
            assert n2 == n and strings(c, table) == report_counts(fixed, thr, dis), (c.name, thr, dis)


@pytest.mark.parametrize("seed", range(7000, 7000 + int(os.environ.get("NB200_FUZZ_CASES", "12"))))
def test_sweep_cases_sit_near_a_switch(seed):
    c = U.sweep_case(seed)
    kind = c.claims["kind"]
    if kind == "token":
        F, nf = c.claims["F"], c.claims["max_nf"]
        assert min(abs(F - s) for s in (127, 128, 511, 512, 32767, 32768)) <= 2
        assert abs(nf - (3 * U.per_key(F) + 1)) <= 2 and c.max_nf() == nf
    elif kind == "group":
        assert abs(c.largest_group() - U.LOCAL_SORT_MAX) <= 2
    elif kind == "general":
        for u in {r[1] for r in c.rows}:
            rows = [r for r in c.rows if r[1] == u]
            assert abs(len(rows) - U.SMALL_ROWS) <= 2
            assert abs(sum(len(r[2].split(",")) for r in rows) - U.SMALL_NAMES) <= 2
    else:
        C, D = c.claims["C"], c.claims["D"]
        assert min(abs(D - (1 << k)) for k in range(9, 14)) <= 2 and min(abs(C - (1 << k)) for k in range(4, 9)) <= 2
        assert len(np.unique(c.key >> np.uint64(32))) == C and len(np.unique(_list_codes(c))) == D
