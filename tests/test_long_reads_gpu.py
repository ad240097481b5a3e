"""The long end of the read range (161-500 bases) against the C oracle, bit for bit: lengths at every 32-base word
boundary with N bases on the N-mask word edges, Smith-Waterman near the top of its s16 range, reads that overhang the
first and last reference by up to 480 bases, 2 x 500 and 28 + 500 pairs, a seeded long-read fuzz, and the streaming
pipeline where a long read shrinks a slab that already holds more short reads than the long read's slab can take."""
import json
import os
import struct
import sys
from collections import Counter
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from nimble_b200 import frontend, synth
from oracle import oracle as O
from helpers import diff_results, oracle_counts, table_tuple, to_concat
from test_align_edge_gpu import _run_in_subprocess, both
from test_fastq_counts_gpu import _check, _write_fastq
from test_oracle_align import lib_of, rc
from test_probe_thread_gpu import thread_vs_warp

pytestmark = pytest.mark.gpu

ACGT = np.frombuffer(b"ACGT", np.uint8)


@pytest.fixture(scope="module")
def engine1():
    """Libraries built on one host thread, so the thread and warp probes read the same table (equal probe counters)."""
    import nimble_b200
    eng = nimble_b200.Engine(0, host_threads=1)
    yield eng
    eng.close()


def _draw(rng, codes, L):
    """A random L-base window of a random allele, as a mutable list of bases."""
    c = codes[int(rng.integers(0, len(codes)))]
    a = int(rng.integers(0, len(c) - L + 1))
    return list(ACGT[c[a:a + L]].tobytes().decode())


def _substitute(s, i):
    s[i] = "ACGT"[("ACGT".index(s[i]) + 1) % 4] if s[i] != "N" else "A"


# ---- 1. lengths at word boundaries ----------------------------------------------------------------------------------

def _groups(k):
    return [(k - 1, k, k + 1), (31, 32, 33), (63, 64, 65), (159, 160, 161), (175, 176, 177), (191, 192, 193),
            (255, 256, 257), (319, 320, 321), (383, 384, 385), (447, 448, 449), (479, 480, 481), tuple(range(495, 501))]


N_POS = [0] + [p for w in range(32, 481, 32) for p in (w - 1, w)]       # first and last base of every N-mask word


def rc_n(s):
    """Reverse complement that keeps N bases."""
    return s[::-1].translate(str.maketrans("ACGTN", "TGCAN"))


def _sweep_case(k):
    """Reads of every length of _groups(k), 24 each: exact, one substitution anywhere, one at the first / last / middle
    base (so reads of k + 1 bases keep one k-mer and go to SW), N bases on word edges and at L - 1, several
    substitutions, a substitution beside an N; a third reverse-complemented.  150 alleles per founder: shared k-mers
    fall in classes of more than four words, so the thread probe also lists reads for the warp form."""
    cfg = {"group_on": "gene"} if k == 31 else {}
    lib, codes = synth.allele_family_library(n_founders=3, alleles_per_founder=150, length=1500, snps_mean=6, seed=600 + k,
                                             config=cfg, extra_columns=k == 31)
    rng = np.random.default_rng(601 + k)
    reads, group_of = [], []
    for g, lens in enumerate(_groups(k)):
        for L in lens:
            for j in range(24):
                s = _draw(rng, codes, L)
                kind = j % 6
                if kind == 1:
                    _substitute(s, int(rng.integers(0, L)))
                elif kind == 2:
                    _substitute(s, (0, L - 1, L // 2, 0)[j // 6])
                elif kind == 3:
                    pos = [p for p in N_POS if p < L] + [L - 1]
                    for p in rng.choice(pos, size=min(len(pos), int(rng.integers(1, 4))), replace=False):
                        s[int(p)] = "N"
                elif kind == 4:
                    for p in rng.integers(0, L, size=int(rng.integers(2, 5))):
                        _substitute(s, int(p))
                elif kind == 5:
                    _substitute(s, int(rng.integers(0, L)))
                    s[int(rng.integers(0, L))] = "N"
                s = "".join(s)
                reads.append(rc_n(s) if rng.random() < 1 / 3 else s)
                group_of.append(g)
    key = synth.barcodes_10x(len(reads), n_cells=20, seed=602 + k)
    return lib, reads, key, np.array(group_of)


@pytest.mark.parametrize("k", [20, 31, 32])
def test_length_sweep_thread_and_warp_probe(engine1, k):
    """Thread probe and NB200_PROBE_WARP=1: both equal the oracle (records, features, table, dropped_empty) and each
    other, probe counters included; every length group went through Smith-Waterman."""
    lib, reads, key, group_of = _sweep_case(k)
    listed = thread_vs_warp(engine1, lib, reads, key, k=k)
    assert listed > 0                                    # reads the thread probe left to the warp form
    assert engine1.timing()["sw_items"] > 0
    lo = O.Library(lib, k=k)
    ro, _ = O.align(lo, to_concat(reads))
    for g, lens in enumerate(_groups(k)):
        assert ro["n_sw"][group_of == g].sum() > 0, lens


WIDE_SWEEP = r"""
import nimble_b200
from test_align_edge_gpu import both
from test_long_reads_gpu import _sweep_case
eng = nimble_b200.Engine(0)
for k in (20, 31, 32):
    lib, reads, key, _ = _sweep_case(k)
    lo, ro, fo, _ = both(eng, lib, reads, key=key, k=k)
    assert ro["n_sw"].sum() > 200 and eng.timing()["sw_items"] > 0
print("sub-ok")
"""


def test_length_sweep_wide_path():
    """NB200_NARROW_CAP=0 sends every read with a hit through wide_kernel: same answers on the whole sweep."""
    _run_in_subprocess({"NB200_NARROW_CAP": "0"}, WIDE_SWEEP)


# ---- 2. Smith-Waterman near the s16 ceiling, long windows in dedupe --------------------------------------------------

SW_LENS = (177, 256, 300, 383, 449, 480, 500)


def _sw_case():
    """Four 1500-base founders.  Per founder: the founder F, an allele with a SNP far from every read, and per read
    length L (reads start at S): T_L with a SNP just past the read's end (a band window that differs from F's only in
    its last 16 bases) and D_L with a SNP at read base L - 20, where the read carries substitutions at L - 21 and L - 19:
    every k-mer over the SNP also covers a substitution, so D_L stays a candidate and scores one mismatch below F, in
    a window that equals F's for the first L - 28 bases."""
    rng = np.random.default_rng(700)
    S = 200
    seqs, names, reads, kinds = [], [], [], []

    def snp(s, p):
        t = list(s)
        _substitute(t, p)
        return "".join(t)

    for f in range(4):
        F = "".join(rng.choice(list("ACGT"), size=1500))
        seqs += [F, snp(F, 1450)]
        names += ["F%d" % f, "F%d-far" % f]
        for L in SW_LENS:
            seqs += [snp(F, S + L + 3), snp(F, S + L - 20)]
            names += ["F%d-T%03d" % (f, L), "F%d-D%03d" % (f, L)]

        def add(s, kind):
            reads.append(s)
            kinds.append(kind)
            reads.append(rc(s))
            kinds.append(kind + "-rc")

        add(F[S:S + 500], "exact500")
        add(F[S + 700:S + 1200], "exact500")
        for p in (0, 499):
            add(snp(F[S:S + 500], p), "end-sub500")
        for L in SW_LENS:
            r = list(F[S:S + L])
            _substitute(r, L - 21)
            _substitute(r, L - 19)
            add("".join(r), "dedupe")
            add(F[S + 1:S + 1 + L], "exact")
            for n_mm in (1, 2, 3):
                r = list(F[S:S + L])
                for p in rng.choice(L, size=n_mm, replace=False):
                    _substitute(r, int(p))
                add("".join(r), "mismatch")
        for d in list(range(1, 13)):
            for a in (25, 250, 470):
                src = F[S:S + 500 + d]
                add(src[:a] + src[a + d:], "del%d" % d)                       # deletion of d bases, 500 left
                ins = "".join(rng.choice(list("ACGT"), size=d))
                add((F[S:S + a] + ins + F[S + a:S + 500])[:500], "ins%d" % d)   # insertion of d bases
    return lib_of(seqs, names, num_mismatches=0, max_hits_to_report=40), reads, np.array(kinds)


def test_sw_near_s16_ceiling(engine):
    """500-base exact reads score 500 with 0 edits (all k-mers hit: no SW); 500-base reads with a substitution at the
    first or last base go through SW at V = 64 * 499, the largest V an alignment reaches, and score 499 with 0 edits;
    1-3 mismatches and indels of 1-12 bases near the start, middle and end; the long windows of the dedupe reads."""
    lib, reads, kinds = _sw_case()
    assert max(map(len, reads)) == 500
    key = synth.barcodes_10x(len(reads), n_cells=4, seed=701)
    lo, ro, fo, _ = both(engine, lib, reads, key=key, k=20)
    tm = engine.timing()
    fwd = np.array([0 if not k.endswith("-rc") else 1 for k in kinds])
    sc = ro["score"][np.arange(len(reads)), fwd]
    ed = ro["edits"][np.arange(len(reads)), fwd]
    ex = np.char.startswith(kinds, "exact500")
    assert ex.sum() == 16 and (sc[ex] == 500).all() and (ed[ex] == 0).all() and (ro["n_sw"][ex] == 0).all()
    es = np.char.startswith(kinds, "end-sub500")
    assert es.sum() == 16 and (sc[es] == 499).all() and (ed[es] == 0).all() and (ro["n_sw"][es] > 0).all()
    sw = ~np.char.startswith(kinds, "exact")
    assert (ro["n_sw"][sw] > 0).all()
    dd = np.char.startswith(kinds, "dedupe")
    assert (ro["reason"][dd] == 0).all()                  # called: F and the alleles that share its window, not D_L
    # identical windows of F, F-far and T_L were aligned once: fewer distinct windows than SW items
    assert 0 < tm["sw_pairs"] < tm["sw_items"]


# ---- 3. reads that overhang the first and last reference -------------------------------------------------------------

@pytest.mark.parametrize("k", [20, 31])
def test_reference_overhangs(engine, k):
    """Reads of 300-500 bases that start up to 480 bases before the first base of a reference or end up to 480 bases
    after its last base, on the first and last reference in internal (feature-name) order, which are not first and last
    in the input; both orientations.  The band window then lies in the padding around the reference."""
    rng = np.random.default_rng(800 + k)
    names = ["M-mid-1", "Z-last", "B-second", "A-first", "M-mid-2"]
    seqs = ["".join(rng.choice(list("ACGT"), size=1200)) for _ in names]
    lib = lib_of(seqs, names, score_percent=0.0, score_threshold=10, score_filter=10)
    reads, expect_sw = [], []
    for name in ("A-first", "Z-last"):
        R = seqs[names.index(name)]
        for L in (300, 333, 400, 480, 500):
            for o in sorted({1, 8, 9, 64, 200, L - 60, L - 2 * k, min(480, L - k - 1)}):
                junk = "".join(rng.choice(list("ACGT"), size=o))
                for s in (junk + R[:L - o], R[len(R) - (L - o):] + junk):
                    assert len(s) == L
                    reads += [s, rc(s)]
                    expect_sw += [True, True]
    key = synth.barcodes_10x(len(reads), n_cells=3, seed=801)
    lo, ro, fo, _ = both(engine, lib, reads, key=key, k=k)
    assert (ro["n_sw"][np.array(expect_sw)] > 0).all()
    assert (ro["reason"] == 0).sum() > len(reads) // 2


# ---- 4. paired-end at the top of the range ----------------------------------------------------------------------------

def _long_pairs(codes, n, seed):
    """2 x 500 pairs, and 28-40 + 450-500 pairs in both mate assignments; fragments up to 1100 bases, mate 2
    reverse-complemented, half of the pairs swapped, 0.5 % substitutions and some N."""
    rng = np.random.default_rng(seed)
    r1, r2 = [], []
    for i in range(n):
        kind = i % 3
        la, lb = (500, 500) if kind == 0 else (int(rng.integers(28, 41)), int(rng.integers(450, 501)))
        if kind == 2:
            la, lb = lb, la
        c = codes[int(rng.integers(0, len(codes)))]
        F = int(rng.integers(max(la, lb), min(len(c), 1100) + 1))
        a = int(rng.integers(0, len(c) - F + 1))
        frag = ACGT[c[a:a + F]].tobytes().decode()
        m = [list(frag[:la]), list(rc(frag[F - lb:]))]
        for s in m:
            for p in np.nonzero(rng.random(len(s)) < 0.005)[0]:
                _substitute(s, int(p))
            if rng.random() < 0.1:
                s[int(rng.integers(0, len(s)))] = "N"
        if rng.random() < 0.5:
            m.reverse()
        r1.append("".join(m[0]))
        r2.append("".join(m[1]))
    return r1, r2


PAIR_CFGS = [{"intersect_level": 0}, {"intersect_level": 1}, {"intersect_level": 2}, {"require_valid_pair": True}]


@pytest.mark.parametrize("strand", ["unstranded", "none"])
@pytest.mark.parametrize("cfg", PAIR_CFGS, ids=[str(c) for c in PAIR_CFGS])
def test_pairs_at_500_bases(engine, cfg, strand):
    """Compact and full wire forms give the same records and table, and both equal the oracle's."""
    lib, codes = synth.allele_family_library(n_founders=4, alleles_per_founder=8, length=1500, snps_mean=10, seed=900,
                                             config=dict(cfg, num_mismatches=1))
    r1, r2 = _long_pairs(codes, 1500, 901)
    key = synth.barcodes_10x(len(r1), n_cells=10, seed=902)
    lg = engine.load_library(lib, strand_filter=strand)
    got = []
    for compact in (True, False):
        p1, p2 = engine.pack(r1, compact=compact), engine.pack(r2, compact=compact)
        assert p1.compact == compact and p1.words == 16
        got.append(engine.align(lg, p1, p2, key=key, per_read=True))
    (tc, rc_, fc), (tf, rf, ff) = got
    assert not diff_results(rf, ff, rc_, fc)
    assert table_tuple(tc.cell, tc.count, tc.feat_off, tc.feat_ids) == table_tuple(tf.cell, tf.count, tf.feat_off, tf.feat_ids)
    lo, ro, fo, _ = both(engine, lib, r1, r2, key=key, strand=strand)
    assert ro["n_sw"].sum() > 100 and (ro["reason"] == 0).sum() > 100


# ---- 5. long-read fuzz ----------------------------------------------------------------------------------------------

def _long_fuzz_case(seed):
    """_fuzz_case's shape (every config knob, k, strand filter, N bases, ragged lengths, barcodes) with reads of
    150-500 bases and references long enough for them."""
    rng = np.random.default_rng(seed)
    k = int(rng.choice([11, 16, 20, 20, 25, 31, 32]))
    cfg = {
        "score_threshold": int(rng.choice([0, 20, 45, 80])), "score_filter": int(rng.choice([0, 25, 60])),
        "score_percent": float(rng.choice([0.0, 0.25, 0.5, 0.8, 1.0])), "num_mismatches": int(rng.choice([0, 0, 1, 2, 5])),
        "discard_multiple_matches": bool(rng.random() < 0.2), "intersect_level": int(rng.choice([0, 1, 2])),
        "discard_multi_hits": int(rng.choice([0, 0, 0, 1, 3])), "require_valid_pair": bool(rng.random() < 0.3),
        "max_hits_to_report": int(rng.choice([1, 2, 5, 10, 17])),
    }
    grouped = rng.random() < 0.3
    if grouped:
        cfg["group_on"] = "gene"
    rl = int(rng.integers(150, 501))
    lib, codes = synth.allele_family_library(n_founders=int(rng.integers(1, 6)), alleles_per_founder=int(rng.integers(1, 30)),
                                             length=int(rng.integers(rl + 60, 1600)), snps_mean=float(rng.choice([0.0, 4.0, 12.0])),
                                             seed=seed, config=cfg, extra_columns=grouped)
    min_len = min(len(c) for c in codes)
    n = int(rng.integers(200, 1500))
    err = float(rng.choice([0.0, 0.005, 0.02]))
    if rng.random() < 0.5:
        r1, r2, truth = synth.sample_pairs(codes, n, read_len=rl, insert_mean=min(min_len, int(rl * rng.uniform(1.0, 2.5))),
                                           insert_sd=40, err_rate=err, off_target=0.15, seed=seed + 1)
    else:
        (r1, truth), r2 = synth.sample_reads(codes, n, read_len=rl, err_rate=err, off_target=0.15,
                                             rc_frac=float(rng.choice([0.1, 0.5])), seed=seed + 1), None
    reads1 = [bytes(r).decode() for r in r1]
    reads2 = [bytes(r).decode() for r in r2] if r2 is not None else None
    for i in rng.choice(n, size=n // 20, replace=False):
        s = list(reads1[i]); s[int(rng.integers(0, len(s)))] = "N"; reads1[i] = "".join(s)
    for i in rng.choice(n, size=n // 10, replace=False):
        reads1[i] = reads1[i][:int(rng.integers(0, len(reads1[i]) + 1))]
        if reads2 is not None and rng.random() < 0.5:
            reads2[i] = reads2[i][int(rng.integers(0, len(reads2[i]))):]
    key = None
    if rng.random() < 0.8:
        key = synth.barcodes_10x(n, n_cells=int(rng.integers(1, 30)), reads_per_umi=float(rng.choice([1.0, 3.0])), seed=seed + 2,
                                 truth=truth if rng.random() < 0.5 else None)
        key[rng.random(n) < 0.03] = np.uint64(0xFFFFFFFFFFFFFFFF)
    strand = str(rng.choice(["unstranded", "fiveprime", "threeprime", "none"]))
    thr = float(rng.choice([0.0, 0.05, 0.2]))
    return lib, reads1, reads2, key, k, strand, thr, bool(rng.random() < 0.15)


@pytest.mark.parametrize("seed", range(5000, 5000 + int(os.environ.get("NB200_FUZZ_CASES", "12"))))
def test_long_read_fuzz(engine, seed):
    lib, r1, r2, key, k, strand, thr, disable = _long_fuzz_case(seed)
    both(engine, lib, r1, r2, key=key, k=k, strand=strand, threshold=thr, disable=disable)


# ---- 6. streaming slabs that shrink for a long read -------------------------------------------------------------------

def slab_room(L):
    """Reads one streaming slab holds when its longest read has L bases: 2^17, or fewer when the packed stride of L
    bases (stream.cpp stride_for) times 2^17 reads would overflow the slab's 64-byte-per-read sequence buffer."""
    w = max(1, (L + 31) // 32)
    return min(1 << 17, (1 << 23) // ((12 * w + 15) & ~15))


def _schedule(long_lens, short=60):
    """Read lengths such that before every long read L the walker's task holds slab_room(L) short reads, so it is cut
    before the long read; the slab that starts with the long read is then filled to slab_room(L) with short reads, and
    the next one starts short again."""
    lens = []
    for L in long_lens:
        assert slab_room(L) < slab_room(short)
        lens += [short] * slab_room(L) + [L] + [short] * (slab_room(L) - 1)
    return lens + [short] * 777


def _reads_of(codes, lens, seed):
    """One read per entry of lens, sampled per run of equal lengths: list of ASCII matrices in input order."""
    out, i = [], 0
    while i < len(lens):
        j = i
        while j < len(lens) and lens[j] == lens[i]:
            j += 1
        out.append(synth.sample_reads(codes, j - i, read_len=lens[i], seed=seed + i)[0])
        i = j
    return out


def _bam_path(tmp_path, name, parts, key, flags=None):
    """Unaligned BAM (file_bench.bam_records per run of equal lengths); parts = [matrix] or [(mate 1, mate 2)] with the
    pair's records back to back under one name, flags (mate 1, mate 2)."""
    import file_bench
    raw, n = [], 0
    for p in parts:
        if flags is None:
            raw.append(file_bench.bam_records(p, key[n:n + len(p)], n))
            n += len(p)
            continue
        recs = []
        for m, fl in zip(p, flags):
            a = np.frombuffer(file_bench.bam_records(m, key[n:n + len(m)], n), np.uint8).reshape(len(m), -1).copy()
            a[:, 18:20] = np.frombuffer(struct.pack("<H", fl), np.uint8)
            recs.append(a)
        raw.append(np.concatenate(recs, axis=1).tobytes())
        n += len(p[0])
    path = str(tmp_path / name)
    with open(path, "wb") as f, ThreadPoolExecutor(8) as ex:
        file_bench.bgzf_append(f, b"BAM\x01" + struct.pack("<i", 0) + struct.pack("<i", 0) + b"".join(raw), ex)
        f.write(file_bench.BGZF_EOF)
    return path


def _stream_lib(tmp_path, seed):
    lib, codes = synth.allele_family_library(n_founders=6, alleles_per_founder=12, length=1200, snps_mean=10, seed=seed)
    path = str(tmp_path / "lib.json")
    with open(path, "w") as f:
        json.dump(lib, f)
    return lib, codes, path


def _check_per_read_tsv(path, lo, ro, fo):
    """Every row of a tagged per-read TSV is the oracle's call for its read (features, four scores), called reads only,
    once each, in input order."""
    rows = open(path).read().split("\n")
    assert rows[0].split("\t")[:2] == ["nimble_features", "nimble_score"] and rows[-1] == ""
    called = np.nonzero(ro["n_feat"])[0]
    assert len(rows) - 2 == len(called) > 0
    for row, i in zip(rows[1:-1], called):
        f = row.split("\t")
        assert f[6] == "r%09d" % i
        assert f[0] == ",".join(lo.features[j] for j in fo[i, :ro["n_feat"][i]]), i
        assert f[2:6] == [str(int(x)) for x in ro["score"][i]], i


def test_stream_single_end_bam_slab_shrinks(engine, tmp_path):
    """(a) single-end BAM (the segment path): long reads of 161-500 bases each arrive when the task holds more short
    reads than slab_room(L); per-read TSV rows against the oracle.  (d) align --counts on the same file against
    oracle_counts."""
    lib, codes, lib_path = _stream_lib(tmp_path, 1000)
    lens = _schedule([161, 257, 385, 449, 500])
    parts = _reads_of(codes, lens, 1001)
    key = synth.barcodes_10x(len(lens), n_cells=300, seed=1002)
    bam = _bam_path(tmp_path, "se.bam", parts, key)
    out, cnt = str(tmp_path / "se.tsv"), str(tmp_path / "se.counts.tsv")
    assert frontend.align(lib_path, out, [bam], 4, "unstranded", "", None, engine=engine) == 0
    lo = O.Library(lib, k=20)
    r1 = [bytes(r).decode() for p in parts for r in p]
    assert [len(r) for r in r1] == lens
    ro, fo = O.align(lo, to_concat(r1))
    _check_per_read_tsv(out, lo, ro, fo)
    long_ = np.nonzero(np.array(lens) > 160)[0]
    assert len(long_) == 5 and (ro["n_feat"][long_] > 0).all()          # the long reads have rows of their own
    # (d)
    assert frontend.align(lib_path, None, [bam], 4, "unstranded", "", None, engine=engine, counts=cnt) == 0
    cell, count, off, ids, dropped = oracle_counts(lo, ro, fo, key)
    want = sorted((",".join(lo.features[j] for j in ids[off[i]:off[i + 1]]), int(count[i]), synth.unpack_barcode(cell[i], 16))
                  for i in range(len(cell)))
    got = []
    for line in open(cnt).read().splitlines():
        f, c, cb = line.split("\t")
        got.append((f, int(c), cb))
    assert len(want) > 1000 and sorted(got) == want
    o3 = engine.align_files_counts([bam], [engine.load_library(lib_path)], [str(tmp_path / "se2.tsv")])
    assert o3[0][1:] == (len(want), dropped)


def test_stream_paired_bam_one_long_mate(engine, tmp_path):
    """(b) paired BAM: the task is cut before a pair whose mate 1 or mate 2 has 161 or 500 bases."""
    lib, codes, lib_path = _stream_lib(tmp_path, 1100)
    lens = _schedule([161, 500, 500])
    m1 = _reads_of(codes, lens, 1101)
    m2 = _reads_of(codes, [60] * len(lens), 1102)
    parts, a = [], 0
    for q, p in enumerate(m1):                 # split m2 along m1's runs; the middle long pair has its long read as mate 2
        b = a + len(p)
        mates = (p, m2[0][a:b]) if not (len(p) == 1 and q == 3) else (m2[0][a:b], p)
        parts.append(mates)
        a = b
    assert sum(max(x.shape[1], y.shape[1]) == 500 and x.shape[1] == 60 for x, y in parts) == 1
    key = synth.barcodes_10x(len(lens), n_cells=300, seed=1103)
    bam = _bam_path(tmp_path, "pe.bam", parts, key, flags=(77, 141))
    out = str(tmp_path / "pe.tsv")
    assert frontend.align(lib_path, out, [bam], 4, "unstranded", "", None, engine=engine) == 0
    lo = O.Library(lib, k=20)
    r1 = [bytes(r).decode() for x, _ in parts for r in x]
    r2 = [bytes(r).decode() for _, y in parts for r in y]
    ro, fo = O.align(lo, to_concat(r1), to_concat(r2))
    _check_per_read_tsv(out, lo, ro, fo)


def test_stream_fastq_slab_shrinks(engine, tmp_path):
    """(c) plain single-end FASTQ: the bulk table (features, reads) equals the oracle's calls."""
    lib, codes, lib_path = _stream_lib(tmp_path, 1200)
    lens = _schedule([193, 449, 481])
    r1 = [bytes(r).decode() for p in _reads_of(codes, lens, 1201) for r in p]
    fq = str(tmp_path / "in.fastq")
    _write_fastq(fq, [("q%d" % i, s, "F" * len(s)) for i, s in enumerate(r1)])
    out = str(tmp_path / "fq.tsv")
    assert frontend.align(lib_path, out, [fq], 4, "unstranded", "", None, engine=engine) == 0
    lo = O.Library(lib, k=20)
    ro, fo = O.align(lo, to_concat(r1))
    want = Counter(",".join(lo.features[j] for j in fo[i, :ro["n_feat"][i]]) for i in np.nonzero(ro["n_feat"])[0])
    rows = open(out).read().splitlines()
    assert rows[0] == "nimble_features\tnimble_score"
    got = Counter({r.split("\t")[0]: int(r.split("\t")[1]) for r in rows[1:]})
    assert len(rows) - 1 == len(want) and got == want


def test_stream_fastq_to_counts_long_r2(engine, tmp_path):
    """(e) fastq-to-counts: R2 of 450-500 bases (at slab cuts, and in a closing run of long pairs), R1 tails of 0-100
    bases after the 16-base barcode and 12-base UMI: the counts bytes equal fastq-to-bam + align --counts."""
    lib, codes, lib_path = _stream_lib(tmp_path, 1300)
    rng = np.random.default_rng(1301)
    lens2 = _schedule([450, 500]) + [int(x) for x in rng.integers(450, 501, size=3000)]
    r2 = [bytes(r).decode() for p in _reads_of(codes, lens2, 1302) for r in p]
    n = len(r2)
    tail = synth.sample_reads(codes, n, read_len=100, seed=1303)[0]
    tl = rng.integers(0, 101, size=n)
    wl, cb, q = synth.barcode_workload(n, n_whitelist=2000, n_cells=300, err_rate=0.01, off_whitelist=0.01, seed=1304)
    umi = ACGT[rng.integers(0, 4, size=(4000, 12))][rng.integers(0, 4000, size=n)]
    s1 = [cb[i].tobytes().decode() + umi[i].tobytes().decode() + tail[i, :tl[i]].tobytes().decode() for i in range(n)]
    q1 = ["".join(chr(33 + int(x)) for x in q[i]) + "F" * (12 + int(tl[i])) for i in range(n)]
    f1, f2, wlp = str(tmp_path / "R1.fastq"), str(tmp_path / "R2.fastq"), str(tmp_path / "wl.txt")
    _write_fastq(f1, [("p%d" % i, s1[i], q1[i]) for i in range(n)])
    _write_fastq(f2, [("p%d" % i, r2[i], "F" * len(r2[i])) for i in range(n)])
    with open(wlp, "w") as f:
        f.write("\n".join(bytes(w).decode() for w in wl) + "\n")
    st, o3, _ = _check(engine, tmp_path, f1, f2, wlp, [engine.load_library(lib_path)], tag="long")
    assert st["total_pairs"] == n and st["no_remaining_seq"] > 0 and o3[0][0] > 10_000 and o3[0][1] > 100
