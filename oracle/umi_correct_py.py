"""ORACLE (test infrastructure, never shipped, never on the product path).

UMI correction (`--correct-umis`, DESIGN.md §2.12) restated at string level, as the rule reads.  It runs on the rows
before `oracle/a6_py.py: report_counts`, which is unchanged.  The rule is modelled on Cell Ranger's `correct_umis`
(Cell Ranger 2.x-3.x), recalled and not pinned by any fixture: the CUDA path is checked against this file, nothing more.
"""
from __future__ import annotations

from oracle.a6_py import _is_null

_UMI_CODE_BASES = "ACGTN"


def _counts_row(cb, umi, feats, score):
    """a6_py.merge_rows' filter: the rows that reach the UMI stage."""
    if _is_null(cb) or _is_null(umi) or _is_null(feats) or _is_null(score):
        return False
    return cb != "" and umi != "" and feats != ""


def correct_umis(rows):
    """rows: (cb, umi, features_string, score).  Per cell, n(cb, u) = rows that count with UMI u.  A UMI of 1..13 bases
    over ACGTN is rewritten to the maximum of (n, UMI string) over itself and every present UMI of the same cell that is
    it with one position replaced by one of A C G T other than the base there; every target from the uncorrected counts
    (one step, no chains followed).  Other UMIs, and rows that do not count, are left as they are.
    Returns (rows in input order, keys (cb, umi) corrected)."""
    n = {}
    for cb, umi, feats, score in rows:
        if _counts_row(cb, umi, feats, score):
            n[(cb, umi)] = n.get((cb, umi), 0) + 1
    target = {}
    for (cb, u), cnt in n.items():
        best = (cnt, u)
        if 1 <= len(u) <= 13 and all(ch in _UMI_CODE_BASES for ch in u):
            for p in range(len(u)):
                for b in "ACGT":
                    if b == u[p]:
                        continue
                    v = u[:p] + b + u[p + 1:]
                    if (cb, v) in n:
                        best = max(best, (n[(cb, v)], v))      # str order of ACGTN is byte order
        target[(cb, u)] = best[1]
    out = [(cb, target[(cb, umi)], feats, score) if _counts_row(cb, umi, feats, score) else (cb, umi, feats, score)
           for cb, umi, feats, score in rows]
    return out, sum(1 for k, t in target.items() if k[1] != t)
