"""UMI correction (`--correct-umis`, DESIGN.md §2.12) without a GPU: the oracle's rule case by case, the base-5 neighbour
arithmetic of the correction kernel against string substitution, the Python mirror of the UMI code, and the flag on the
three commands that take it."""
import random

import numpy as np
import pytest

from nimble_b200 import __main__ as cli
from nimble_b200 import _lib, frontend
from oracle.a6_py import report_counts
from oracle.umi_correct_py import correct_umis


def _rows(spec, feats="A", cell="c1"):
    """spec: [(umi, n)] -> n rows each, in the order given"""
    return [(cell, u, feats, 1.0) for u, k in spec for _ in range(k)]


def _umis(rows):
    return [r[1] for r in rows]


def test_one_read_umi_merges_into_five_read_neighbour():
    out, n = correct_umis(_rows([("ACGTACGTACGT", 5), ("ACGTACGAACGT", 1)]))
    assert n == 1 and set(_umis(out)) == {"ACGTACGTACGT"}
    assert report_counts(out)[0] == [("A", 1, "c1")]


def test_equal_counts_byte_greater_wins():
    out, n = correct_umis(_rows([("AAGA", 1), ("AATA", 1)]))              # G < T
    assert n == 1 and _umis(out) == ["AATA", "AATA"]
    out, n = correct_umis(_rows([("AANA", 1), ("AATA", 1)]))              # N < T: the N position moves to T
    assert n == 1 and _umis(out) == ["AATA", "AATA"]
    out, n = correct_umis(_rows([("AAGA", 1), ("AANA", 1)]))              # G < N, and no UMI is rewritten to an N
    assert n == 0 and _umis(out) == ["AAGA", "AANA"]
    out, n = correct_umis(_rows([("CAAA", 2), ("AAAA", 2), ("GAAA", 2)]))   # three-way tie at one position: G
    assert n == 2 and set(_umis(out)) == {"GAAA"}


def test_chain_is_one_step_from_the_original_counts():
    rows = _rows([("AAAA", 1), ("AAAC", 2), ("AACC", 3)])
    out, n = correct_umis(rows)
    assert n == 2 and _umis(out) == ["AAAC"] + ["AACC"] * 5
    assert report_counts(out)[0] == [("A", 2, "c1")]


def test_other_cells_distance_two_and_other_lengths_stay():
    rows = _rows([("ACGT", 5)], cell="c1") + _rows([("ACGA", 1)], cell="c2")
    assert correct_umis(rows) == (rows, 0)
    rows = _rows([("ACGT", 5), ("ACCA", 1)])                              # Hamming distance 2
    assert correct_umis(rows) == (rows, 0)
    rows = _rows([("ACGT", 5), ("ACG", 1), ("ACGTA", 1)])                 # a shorter and a longer UMI
    assert correct_umis(rows) == (rows, 0)


def test_long_and_non_acgtn_umis_are_untouched():
    rows = _rows([("A" * 14, 5), ("A" * 13 + "C", 1)])                    # 14 bases: not a code
    assert correct_umis(rows) == (rows, 0)
    rows = _rows([("ACGT", 5), ("ACGX", 1), ("acgt", 1)])
    assert correct_umis(rows) == (rows, 0)


def test_rows_that_do_not_count_are_neither_counted_nor_rewritten():
    rows = _rows([("ACGT", 1), ("ACGA", 1)]) + [("c1", "ACGA", "", 1.0), ("c1", "ACGA", "A", float("nan"))]
    out, n = correct_umis(rows)                                          # equal support 1 : 1, T > A
    assert n == 1 and _umis(out) == ["ACGT", "ACGT", "ACGA", "ACGA"]


def test_thresholding_sees_the_merged_rows():
    """20 rows of A on one UMI, 1 row of B on a neighbour.  Apart, both UMIs count.  Merged, B's ratio 1/21 < 0.05 is
    dropped by the thresholding of the merged UMI; without thresholding the merged UMI's rows intersect to nothing."""
    rows = _rows([("ACGTAC", 20)], "A") + _rows([("ACGTAA", 1)], "B")
    assert report_counts(rows) == ([("A", 1, "c1"), ("B", 1, "c1")], 0)
    out, n = correct_umis(rows)
    assert n == 1
    assert report_counts(out) == ([("A", 1, "c1")], 0)
    assert report_counts(out, disable_thresholding=True) == ([], 1)


def _decode(code):
    s = []
    while code:
        q = (code - 1) // 5
        s.append("ACGTN"[code - 5 * q - 1])
        code = q
    return "".join(reversed(s))


def test_neighbour_arithmetic_matches_string_substitution():
    L = _lib.load()
    import ctypes as ct
    oc, ov = (ct.c_uint32 * 52)(), (ct.c_uint32 * 52)()
    rng = random.Random(7)
    for trial in range(3000):
        n = 1 + trial % 13
        u = "".join(rng.choice("ACGTN" if trial % 3 else "ACGT") for _ in range(n))
        code = frontend.umi_code(u)
        assert code is not None and _decode(code) == u
        k = L.nb200_umi_neighbours(code, oc, ov)
        got = [_decode(oc[i]) for i in range(k)]
        want = {u[:p] + b + u[p + 1:] for p in range(n) for b in "ACGT" if b != u[p]}
        assert len(got) == k == len(want) and set(got) == want, u
        assert all(len(g) == n for g in got)
        # the byte-order value sorts the neighbours as their bytes do
        by_value = [g for _, g in sorted(zip(ov[:k], got))]
        assert by_value == sorted(got), u
    for bad in (0, frontend.UMI_CODE_MAX + 1, 0x80000001, 0xFFFFFFFF):
        assert L.nb200_umi_neighbours(bad, oc, ov) == -1


def test_python_umi_code_mirror():
    assert frontend.umi_code("A") == 1 and frontend.umi_code("N") == 5 and frontend.umi_code("AA") == 6
    assert frontend.umi_code("N" * 13) == frontend.UMI_CODE_MAX < 2 ** 31
    for bad in ("", "A" * 14, "ACGX", "acgt"):
        assert frontend.umi_code(bad) is None
    vals = ["ACGT", "ACGT", "A" * 14, "ACG", "X", "A" * 14, "ACGTN"]
    ids = frontend._umi_ids(vals)
    assert ids.dtype == np.uint64
    assert ids[0] == ids[1] == frontend.umi_code("ACGT") and ids[3] == frontend.umi_code("ACG")
    assert ids[2] == ids[5] == frontend.UMI_INTERNED and ids[4] == frontend.UMI_INTERNED | 1   # "AAAA..." < "X"
    assert len(set(ids.tolist())) == 5


@pytest.fixture
def calls(monkeypatch):
    seen = {}

    def rec(name):
        def f(*a, **kw):
            seen[name] = kw
            return 0
        return f
    for name in ("report", "align", "fastq_to_counts"):
        monkeypatch.setattr(cli, name, rec(name))
    return seen


def test_cli_flag_on_the_three_commands(calls):
    cli.main(["report", "-i", "in.tsv", "-o", "out.tsv", "--correct-umis"])
    assert calls["report"]["correct_umis"] is True
    cli.main(["report", "-i", "in.tsv", "-o", "out.tsv"])
    assert calls["report"]["correct_umis"] is False
    for extra, want in ((["--correct-umis"], True), ([], False)):
        with pytest.raises(SystemExit) as e:
            cli.main(["align", "--reference", "lib.json", "--input", "in.bam", "--counts", "c.tsv"] + extra)
        assert e.value.code == 0 and calls["align"]["correct_umis"] is want
        with pytest.raises(SystemExit) as e:
            cli.main(["fastq-to-counts", "--reference", "lib.json", "--r1-fastq", "r1", "--r2-fastq", "r2", "--map", "wl",
                      "--counts", "c.tsv"] + extra)
        assert e.value.code == 0 and calls["fastq_to_counts"]["correct_umis"] is want


def test_cli_align_correct_umis_needs_counts(calls, capsys):
    with pytest.raises(SystemExit) as e:
        cli.main(["align", "--reference", "lib.json", "--input", "in.bam", "--output", "o.tsv", "--correct-umis"])
    assert e.value.code == 2 and "--correct-umis needs --counts" in capsys.readouterr().err
    assert "align" not in calls
