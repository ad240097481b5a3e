"""UMI correction on the GPU (`--correct-umis`, DESIGN.md §2.12): `report` against the oracle (native and Python TSV
handling) in three UMI shapes and at over a million distinct (cell, UMI) keys; `align --counts` and `fastq-to-counts`
byte for byte against their two-step routes with the flag; the in-memory entries refuse it."""
import ctypes as ct
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from nimble_b200 import _lib, frontend, synth
from nimble_b200._lib import EINVAL
from oracle.a6_py import report_counts
from oracle.umi_correct_py import correct_umis

pytestmark = pytest.mark.gpu


def _read(p):
    with open(p, "rb") as f:
        return f.read()


def _write_tsv(path, rows):
    with open(path, "w") as f:
        f.write("nimble_features\tnimble_score\tr1_CB\tr1_UB\n")
        f.write("".join("%s\t%r\t%s\t%s\n" % (feats, score, cb, umi) for cb, umi, feats, score in rows))


def _expected(rows, threshold=0.05, disable=False):
    fixed, corrected = correct_umis(rows)
    out, dropped = report_counts(fixed, threshold, disable)
    return "".join("%s\t%d\t%s\n" % r for r in out).encode(), len(out), dropped, corrected


def _mutate(rng, umi, alphabet="ACGT"):
    p = int(rng.integers(0, len(umi)))
    b = rng.choice([c for c in alphabet if c != umi[p]])
    return umi[:p] + b + umi[p + 1:]


def _feats(rng, n_names=12):
    k = 1 + int(rng.integers(0, 3) == 0) + int(rng.integers(0, 6) == 0)
    return ",".join("f%02d" % i for i in rng.choice(n_names, size=k, replace=False))


def _shape_10x(rng, n=30_000):
    """12-base UMIs, ~3 rows per molecule, 1 % per-base errors."""
    mols = [("CELL%03d" % rng.integers(0, 150), "".join(rng.choice(list("ACGT"), 12)), _feats(rng)) for _ in range(n // 3)]
    rows = []
    for _ in range(n):
        cb, umi, feats = mols[int(rng.integers(0, len(mols)))]
        for p in range(12):
            if rng.random() < 0.01:
                umi = umi[:p] + rng.choice([c for c in "ACGT" if c != umi[p]]) + umi[p + 1:]
        rows.append((cb, umi, feats if rng.random() < 0.9 else _feats(rng), 1.0 if rng.random() < 0.9 else float(rng.choice([0.5, 2.0, 0.25]))))
    return rows


def _shape_dense(rng, n=6_000):
    """4-base UMIs in 12 cells: most neighbours are present, ties and chains everywhere."""
    return [("CELL%02d" % rng.integers(0, 12), "".join(rng.choice(list("ACGT"), 4)), _feats(rng, 6), 1.0) for _ in range(n)]


def _shape_mixed(rng, n=8_000):
    """6-base UMIs with N bases, 14-base UMIs and UMIs with other bytes (interned, never corrected)."""
    rows = []
    base = ["".join(rng.choice(list("ACGTN"), 6, p=[0.22, 0.22, 0.22, 0.22, 0.12])) for _ in range(600)]
    for _ in range(n):
        x = rng.random()
        if x < 0.1:
            umi = "".join(rng.choice(list("ACGT"), 14))
        elif x < 0.15:
            umi = "".join(rng.choice(list("ACGX"), 5))
        else:
            umi = base[int(rng.integers(0, len(base)))]
            if rng.random() < 0.2:
                umi = _mutate(rng, umi, "ACGTN")
        rows.append(("CELL%02d" % rng.integers(0, 20), umi, _feats(rng, 8), 1.0))
    return rows


@pytest.mark.parametrize("shape", ["10x", "dense", "mixed"])
def test_report_against_oracle(engine, tmp_path, shape, capsys):
    rng = np.random.default_rng({"10x": 1, "dense": 2, "mixed": 3}[shape])
    rows = {"10x": _shape_10x, "dense": _shape_dense, "mixed": _shape_mixed}[shape](rng)
    tsv = str(tmp_path / "in.tsv")
    _write_tsv(tsv, rows)
    for thr, dis in ((0.05, False), (0.2, False), (0.05, True)):
        want, n_out, dropped, corrected = _expected(rows, thr, dis)
        assert corrected > 0
        got = str(tmp_path / "native.tsv")
        assert engine.report_file(tsv, got, thr, dis, True) == (len(rows), n_out, dropped, corrected)
        assert _read(got) == want, (shape, thr, dis)
        py = str(tmp_path / "python.tsv")
        capsys.readouterr()
        frontend.report(tsv, py, threshold=thr, disable_thresholding=dis, engine=engine, native=False, correct_umis=True)
        assert _read(py) == want, (shape, thr, dis)
        assert capsys.readouterr().out.splitlines()[:2] == ["Corrected %d UMIs (Hamming distance 1)" % corrected,
                                                            "Dropped %d UMIs due to empty intersections" % dropped]
    # without the flag: the same input counts as before, and no "Corrected" line
    plain = str(tmp_path / "plain.tsv")
    out, dropped = report_counts(rows)
    frontend.report(tsv, plain, engine=engine)
    assert _read(plain) == "".join("%s\t%d\t%s\n" % r for r in out).encode()
    assert capsys.readouterr().out.splitlines()[0] == "Dropped %d UMIs due to empty intersections" % dropped


def test_report_million_keys_against_oracle(engine, tmp_path):
    """1.2 M rows, over a million distinct (cell, UMI) keys (the slot table is sized from the rows), 5 % of them a
    one-substitution copy of another row's UMI."""
    rng = np.random.default_rng(5)
    n = 1_200_000
    codes = rng.integers(0, 4, size=(n, 10))
    alpha = np.frombuffer(b"ACGT", np.uint8)
    umis = [bytes(r).decode() for r in alpha[codes]]
    cells = ["C%04d" % c for c in rng.integers(0, 3000, size=n)]
    src = rng.integers(0, n, size=n)
    copy = np.nonzero(rng.random(n) < 0.05)[0]
    for i in copy:
        j = int(src[i])
        cells[i] = cells[j]
        umis[i] = _mutate(rng, umis[j])
    feats = ["f%02d" % f for f in rng.integers(0, 5, size=n)]
    rows = list(zip(cells, umis, feats, [1.0] * n))
    assert len(set(zip(cells, umis))) > 1_000_000
    tsv, got = str(tmp_path / "big.tsv"), str(tmp_path / "big_counts.tsv")
    _write_tsv(tsv, rows)
    want, n_out, dropped, corrected = _expected(rows)
    assert corrected > 30_000
    assert engine.report_file(tsv, got, 0.05, False, True) == (n, n_out, dropped, corrected)
    assert _read(got) == want


def _bam_with_ub_errors(tmp_path, n_reads, seed):
    import file_bench
    lib, codes = synth.allele_family_library(n_founders=8, alleles_per_founder=20, length=700, snps_mean=10, seed=seed)
    r1, truth = synth.sample_reads(codes, n_reads, read_len=90, seed=seed + 1)
    key = synth.barcodes_10x(n_reads, n_cells=300, seed=seed + 1, truth=truth)
    rng = np.random.default_rng(seed + 2)
    err = np.nonzero(rng.random(n_reads) < 0.04)[0]             # one substitution in the 12-base UB of 4 % of the reads
    flip = rng.integers(1, 4, size=len(err)).astype(np.uint64) << (2 * rng.integers(0, 12, size=len(err))).astype(np.uint64)
    key[err] ^= flip
    lib_path = str(tmp_path / "lib.json")
    with open(lib_path, "w") as f:
        json.dump(lib, f)
    bam = str(tmp_path / "in.bam")
    file_bench.write_bam(bam, r1, key)
    return lib_path, bam


def test_align_counts_equals_align_then_report(engine, tmp_path, capsys):
    lib_path, bam = _bam_with_ub_errors(tmp_path, 200_000, 61)
    lib = engine.load_library(lib_path)
    per_read = str(tmp_path / "per_read.tsv")
    assert frontend.align(lib_path, per_read, [bam], 4, "unstranded", "", None, engine=engine) == 0
    for thr, dis in ((0.05, True), (0.05, False)):           # the default last: the runs below compare with it
        want, got = str(tmp_path / "want.tsv"), str(tmp_path / "got.tsv")
        o_want = engine.report_file(per_read, want, thr, dis, True)
        o_got = engine.align_files_counts([bam], [lib], [got], None, thr, dis, True)
        assert o_got == [o_want] and o_want[3] > 1000, (thr, dis)
        assert _read(got) == _read(want), (thr, dis)
    plain = str(tmp_path / "plain.tsv")
    engine.align_files_counts([bam], [lib], [plain], None)
    assert _read(plain) != _read(got)
    # two contexts on one GPU: rows gathered from both stores before the correction
    got2 = str(tmp_path / "got2.tsv")
    capsys.readouterr()
    assert frontend.align(lib_path, None, [bam], 4, "unstranded", "", None, gpus=[0, 0], counts=got2, correct_umis=True) == 0
    assert _read(got2) == _read(want)
    assert "Corrected %d UMIs (Hamming distance 1)" % o_want[3] in capsys.readouterr().out


def _tenx_with_umi_errors(tmp_path, codes, n, seed):
    """10x pairs as tests/test_fastq_counts_gpu.py draws them (clustered whitelist: reads with several candidates), the
    12-base UMIs drawn from a pool, 5 % of them with one substitution."""
    from test_fastq_counts_gpu import _write_fastq
    rng = np.random.default_rng(seed)
    r2, _ = synth.sample_reads(codes, n, read_len=90, seed=seed + 1)
    tail, _ = synth.sample_reads(codes, n, read_len=62, seed=seed + 2)
    wl_a, cb, q = synth.barcode_workload(n, n_whitelist=2000, n_cells=300, err_rate=0.02, n_rate=0.002, off_whitelist=0.02,
                                         seed=seed + 3, clustered=0.5)
    pool = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, size=(20000, 12))]
    umi = pool[rng.integers(0, len(pool), size=n)].copy()
    err = np.nonzero(rng.random(n) < 0.05)[0]
    pos = rng.integers(0, 12, size=len(err))
    umi[err, pos] = np.frombuffer(b"ACGT", np.uint8)[(np.searchsorted(np.frombuffer(b"ACGT", np.uint8), umi[err, pos])
                                                       + rng.integers(1, 4, size=len(err))) % 4]
    q1 = (rng.integers(2, 41, size=(n, 74)) + 33).astype(np.uint8)
    q2 = (rng.integers(2, 41, size=(n, 90)) + 33).astype(np.uint8)
    s1 = np.concatenate([cb, umi, tail], axis=1)
    qq1 = np.concatenate([(q + 33).astype(np.uint8), q1], axis=1)
    f1, f2 = str(tmp_path / "in_R1.fastq"), str(tmp_path / "in_R2.fastq")
    _write_fastq(f1, [("p%d/1" % i, s1[i].tobytes().decode(), qq1[i].tobytes().decode()) for i in range(n)])
    _write_fastq(f2, [("p%d/2" % i, r2[i].tobytes().decode(), q2[i].tobytes().decode()) for i in range(n)])
    wlp = str(tmp_path / "wl.txt")
    with open(wlp, "w") as f:
        f.write("\n".join(bytes(r).decode() for r in wl_a) + "\n")
    return f1, f2, wlp


def test_fastq_to_counts_equals_fastq_to_bam_then_align_counts(engine, tmp_path):
    lib, codes = synth.allele_family_library(n_founders=8, alleles_per_founder=20, length=700, snps_mean=10, seed=71)
    lib_path = str(tmp_path / "lib.json")
    with open(lib_path, "w") as f:
        json.dump(lib, f)
    f1, f2, wlp = _tenx_with_umi_errors(tmp_path, codes, 300_000, 72)
    L = engine.load_library(lib_path)
    bam, want, got = str(tmp_path / "s.bam"), str(tmp_path / "want.tsv"), str(tmp_path / "got.tsv")
    engine.fastq_to_bam(f1, f2, wlp, bam, 16, 12)
    o_want = engine.align_files_counts([bam], [L], [want], None, 0.05, False, True)
    st, o_got = engine.fastq_to_counts(f1, f2, wlp, [L], [got], 16, 12, 0.05, False, True)
    assert st["n_multi"] > 0 and st["cb_corrected"] > 1000
    assert o_got == o_want and o_want[0][3] > 1000
    assert _read(got) == _read(want)
    got2 = str(tmp_path / "got2.tsv")
    assert frontend.fastq_to_counts(lib_path, f1, f2, wlp, got2, 8, gpus=[0, 0], correct_umis=True) == 0
    assert _read(got2) == _read(want)


def test_in_memory_entries_refuse_correction(engine, tmp_path):
    lib, codes = synth.allele_family_library(n_founders=2, alleles_per_founder=4, length=400, snps_mean=5, seed=81)
    lib_path = str(tmp_path / "lib.json")
    with open(lib_path, "w") as f:
        json.dump(lib, f)
    lg = engine.load_library(lib_path)
    r1, truth = synth.sample_reads(codes, 1000, read_len=90, seed=82)
    key = synth.barcodes_10x(1000, n_cells=10, seed=83, truth=truth)
    p1 = engine.pack(r1)
    s1 = p1.struct()
    c = _lib.Counts()
    L = engine.L
    assert L.nb200_align(engine.ctx, lg.id, ct.byref(s1), None, key.ctypes.data, 0.05, _lib.UMI_CORRECT, None, None, ct.byref(c)) == EINVAL
    assert b"NB200_UMI_CORRECT" in L.nb200_last_error(engine.ctx)
    assert L.nb200_align(engine.ctx, lg.id, ct.byref(s1), None, key.ctypes.data, 0.05, 4, None, None, ct.byref(c)) == EINVAL
    engine.upload(r1, key=key)
    assert L.nb200_align_resident(engine.ctx, lg.id, 0.05, _lib.UMI_CORRECT | _lib.UMI_NO_THRESHOLD, ct.byref(c)) == EINVAL
    # the context stays usable, and flags 0 / 1 mean what they meant
    t0 = engine.align(lg, r1, key=key)
    t1 = engine.align(lg, r1, key=key, disable_thresholding=True)
    assert t0.n_called == t1.n_called > 0
