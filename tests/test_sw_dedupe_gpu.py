"""Deduplication of Smith-Waterman band windows (dedupe_kernel) and the register-streamed query of sw_kernel, read by
read against the C oracle.  Families of alleles are built so that one read's candidates form a segment of a chosen
size whose windows repeat with a chosen period: the number of windows aligned is then known exactly, including for
segments that span several 32-item chunks and duplicates exactly 32 and 33 items apart."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from nimble_b200 import synth
from test_align_edge_gpu import both
from test_long_reads_gpu import rc_n
from test_oracle_align import lib_of, rc

pytestmark = pytest.mark.gpu

BAND = 8
LOOK_BACK = 32
REF_LEN = 1500
OTHER = {"A": "CGTN", "C": "AGTN", "G": "ACTN", "T": "ACGN"}


def roots(classes):
    """Windows aligned for one segment: an item is aligned unless an identical window is among the LOOK_BACK items
    before it."""
    return sum(all(classes[j] != c for j in range(max(0, k - LOOK_BACK), k)) for k, c in enumerate(classes))


def _family(rng, tag, n, period, S, L):
    """A founder F and n - 1 alleles named so that the library orders them F, 1, 2, ...  Allele k differs from F by
    one base outside every read and window of the family (so all are distinct), and allele k with k % period = c > 0
    also at a base of the band margins [S - 8, S) and [S + L, S + L + 8) inside the reference, by a substitution or an
    N: window class c.  Reads inside [S, S + L) hit the same k-mers in every allele."""
    F = "".join(rng.choice(list("ACGT"), size=REF_LEN))
    margins = [p for p in list(range(S - BAND, S)) + list(range(S + L, S + L + BAND)) if 0 <= p < REF_LEN]
    far = 40 if S > 600 else 1440 - n
    assert far + n <= S - BAND or far >= S + L + BAND
    seqs, names = [F], ["%s_%03d" % (tag, 0)]
    for k in range(1, n):
        s = list(F)
        s[far + k] = OTHER[s[far + k]][0]
        c = k % period
        if c:
            p = margins[(c - 1) % len(margins)]
            s[p] = OTHER[F[p]][(c - 1) // len(margins)]
        seqs.append("".join(s))
        names.append("%s_%03d" % (tag, k))
    return seqs, names, F, [k % period for k in range(n)]


def _reads(F, S, L):
    """Four reads of F[S, S + L) that need Smith-Waterman: a substitution or an N at the middle base, as read and
    reverse-complemented."""
    out = []
    for mark in ("sub", "N"):
        r = list(F[S:S + L])
        m = L // 2
        r[m] = "N" if mark == "N" else OTHER[r[m]][1]
        s = "".join(r)
        out += [s, rc_n(s)]
    return out


# (candidates per segment, period of the window classes, read start, read length)
FAMILIES = [(1, 1, 200, 90), (2, 2, 200, 90), (31, 3, 200, 90), (32, 32, 200, 90), (33, 33, 200, 90),
            (64, 32, 200, 90), (70, 33, 200, 90), (67, 5, 200, 90), (40, 7, 0, 90), (40, 7, REF_LEN - 90, 90),
            (33, 32, 200, 176), (33, 32, 200, 177), (70, 33, 200, 177), (65, 2, 100, 500), (34, 33, 0, 500),
            (34, 33, REF_LEN - 500, 500)]


def _case(families):
    rng = np.random.default_rng(4242)
    seqs, names, reads, want_items, want_pairs = [], [], [], 0, 0
    for f, (n, period, S, L) in enumerate(families):
        s, nm, F, classes = _family(rng, "f%02d" % f, n, period, S, L)
        seqs += s
        names += nm
        rs = _reads(F, S, L) * 6                  # many segments of each shape, at varied chunk offsets
        reads += rs
        want_items += len(rs) * n
        want_pairs += len(rs) * roots(classes)
    return lib_of(seqs, names, max_hits_to_report=64), reads, want_items, want_pairs


def test_roots_rule():
    assert roots([0] * 70) == 1
    assert roots([k % 32 for k in range(64)]) == 32
    assert roots([k % 33 for k in range(70)]) == 70


def test_segments_against_oracle(engine):
    """Segments of 1-70 candidates (odd ones with a padding item) across 32-item chunks, windows with N bases and at
    both reference ends, reads of 90, 176, 177 and 500 bases in both orientations: every read equals the oracle, and
    exactly the windows without an identical one among the 32 items before them are aligned."""
    lib, reads, want_items, want_pairs = _case(FAMILIES)
    order = np.random.default_rng(4243).permutation(len(reads))        # interleave the families' segments
    reads = [reads[i] for i in order]
    key = synth.barcodes_10x(len(reads), n_cells=5, seed=4244)
    lo, ro, fo, _ = both(engine, lib, reads, key=key, k=20)
    tm = engine.timing()
    assert (ro["n_sw"] > 0).all()
    assert tm["sw_items"] == want_items
    assert tm["sw_pairs"] == want_pairs


def test_paired_segments_against_oracle(engine):
    """Paired-end: mate 1 as in the single-end case, mate 2 an exact read further along the same founder."""
    fams = [(33, 32, 200, 90), (70, 33, 200, 90), (31, 3, 200, 90), (34, 33, 200, 177)]
    rng = np.random.default_rng(4245)
    seqs, names, r1, r2 = [], [], [], []
    for f, (n, period, S, L) in enumerate(fams):
        s, nm, F, _ = _family(rng, "p%02d" % f, n, period, S, L)
        seqs += s
        names += nm
        for r in _reads(F, S, L):
            r1.append(r)
            r2.append(rc(F[S + L + 20:S + L + 120]))
    key = synth.barcodes_10x(len(r1), n_cells=3, seed=4246)
    lo, ro, fo, _ = both(engine, lib_of(seqs, names, max_hits_to_report=64), r1, r2, key=key, k=20)
    assert (ro["n_sw"] > 0).all()
    assert engine.timing()["sw_pairs"] < engine.timing()["sw_items"]


# Windows aligned for the first 200 000 reads of the cfg2 workload (bench.py make_workload) with one fingerprint pass
# and one look-back pass over global memory, the kernels dedupe_kernel replaced.
CFG2_SW_PAIRS_TWO_PASS = 117_400


def test_cfg2_shaped_batch(engine):
    """A cfg2-shaped batch equals the oracle, and aligns no more windows than the two-pass dedupe did (1 % slack)."""
    lib, codes = synth.allele_family_library(n_founders=40, alleles_per_founder=50, length=1098, snps_mean=15.0, seed=1)
    asc, truth = synth.sample_reads(codes, 200_000, read_len=90, err_rate=0.005, off_target=0.2, rc_frac=0.1, seed=2)
    reads = [bytes(r).decode() for r in asc]
    key = synth.barcodes_10x(len(reads), n_cells=1000, seed=3, truth=truth)
    both(engine, lib, reads, key=key, k=20)
    tm = engine.timing()
    print("cfg2-shaped batch: sw_items %d sw_pairs %d" % (tm["sw_items"], tm["sw_pairs"]))
    assert 0 < tm["sw_pairs"] < tm["sw_items"]
    assert tm["sw_pairs"] <= 1.01 * CFG2_SW_PAIRS_TWO_PASS
