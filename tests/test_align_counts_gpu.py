"""`align --counts` (nb200_align_files_counts / nb200_align_files_counts_multi): reads to the counts TSV in one streaming
pass, the rows of the UMI stage kept on the GPU.  Every case compares the counts file byte for byte with the two-step
route `align` -> `report` on the same input."""
import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "scripts"))

from nimble_b200 import frontend, synth
from nimble_b200._lib import EINVAL, NimbleB200Error
from test_frontend import write_bam

pytestmark = pytest.mark.gpu


def _inputs(tmp_path, n_reads, seed):
    import file_bench
    lib, codes = synth.allele_family_library(n_founders=8, alleles_per_founder=20, length=700, snps_mean=10, seed=seed)
    r1, truth = synth.sample_reads(codes, n_reads, read_len=90, seed=seed + 1)
    key = synth.barcodes_10x(n_reads, n_cells=500, seed=seed + 1, truth=truth)
    lib_path = str(tmp_path / "lib.json")
    with open(lib_path, "w") as f:
        json.dump(lib, f)
    bam = str(tmp_path / "in.bam")
    file_bench.write_bam(bam, r1, key)
    return lib_path, bam


def _two_step(engine, tmp_path, ref, bam, threshold=0.05, disable=False, trim="", tag="ts"):
    """align -> report per library; returns ([per-read TSV paths], [counts paths], [report out3])."""
    libs = ref.split(",")
    out = str(tmp_path / ("%s.tsv" % tag))
    assert frontend.align(ref, out, [bam], 4, "unstranded", trim, None, engine=engine) == 0
    outs = frontend._per_library_paths(out, libs)
    cnts, o3 = [], []
    for i, o in enumerate(outs):
        c = str(tmp_path / ("%s.counts.%d.tsv" % (tag, i)))
        o3.append(engine.report_file(o, c, threshold, disable))
        cnts.append(c)
    return outs, cnts, o3


def _read(p):
    with open(p, "rb") as f:
        return f.read()


def test_counts_single_end_three_slabs_thresholds(engine, tmp_path):
    """300 k reads (three slabs), 500 cells: counts and out3 equal report's for thresholds 0.05, 0.2 and none."""
    lib_path, bam = _inputs(tmp_path, 300_000, 91)
    lib = engine.load_library(lib_path)
    out = str(tmp_path / "ts.tsv")
    assert frontend.align(lib_path, out, [bam], 4, "unstranded", "", None, engine=engine) == 0
    for thr, dis in ((0.05, False), (0.2, False), (0.05, True)):
        want, got = str(tmp_path / "want.tsv"), str(tmp_path / "got.tsv")
        o3_want = engine.report_file(out, want, thr, dis)
        o3_got = engine.align_files_counts([bam], [lib], [got], None, thr, dis)
        assert o3_got == [o3_want] and o3_want[0] > 100_000 and o3_want[1] > 1000, (thr, dis)
        assert _read(got) == _read(want), (thr, dis)


def test_counts_paired_two_libraries_trim(engine, tmp_path):
    """Paired BAM, two libraries, --trim, one call: each library's counts equal the two-step route's, and the per-read
    TSVs written in the same pass equal nb200_align_files'."""
    lib_a, codes = synth.allele_family_library(n_founders=6, alleles_per_founder=10, length=800, snps_mean=8, seed=11)
    lib_b, _ = synth.allele_family_library(n_founders=6, alleles_per_founder=10, length=800, snps_mean=8, seed=11, name_prefix="Mafa")
    pa, pb = str(tmp_path / "liba.json"), str(tmp_path / "libb.json")
    for p, lb in ((pa, lib_a), (pb, lib_b)):
        with open(p, "w") as f:
            json.dump(lb, f)
    n = 40_000
    m1, m2, truth = synth.sample_pairs(codes, n, read_len=120, seed=12)
    key = synth.barcodes_10x(n, n_cells=60, seed=13, truth=truth)
    rng = np.random.default_rng(14)
    q1 = rng.integers(2, 41, size=m1.shape)
    q2 = rng.integers(2, 41, size=m2.shape)
    recs = []
    for i in range(n):
        cb = synth.unpack_barcode(int(key[i]) >> 32, 16)
        ub = synth.unpack_barcode(int(key[i]) & 0xFFFFFF, 12)
        recs.append(("p%d" % i, 77, m1[i].tobytes().decode(), {"CB": cb, "UB": ub}, q1[i]))
        recs.append(("p%d" % i, 141, m2[i].tobytes().decode(), {"CB": cb, "UB": ub}, q2[i]))
    bam = str(tmp_path / "pairs.bam")
    write_bam(bam, recs)
    ref, trim = "%s,%s" % (pa, pb), "70:0.6,90:0.4"
    outs, cnts, o3 = _two_step(engine, tmp_path, ref, bam, trim=trim)
    out2, cnt2 = str(tmp_path / "fused.tsv"), str(tmp_path / "fused_counts.tsv")
    assert frontend.align(ref, out2, [bam], 4, "unstranded", trim, None, engine=engine, counts=cnt2) == 0
    libs = ref.split(",")
    for a, b in zip(outs, frontend._per_library_paths(out2, libs)):
        assert _read(a) == _read(b)
    got = frontend._per_library_paths(cnt2, libs)
    assert got == [str(tmp_path / "fused_counts.liba.tsv"), str(tmp_path / "fused_counts.libb.tsv")]
    for w, g, x in zip(cnts, got, o3):
        assert x[0] > 10_000 and _read(g) == _read(w)


def test_counts_edge_barcodes_and_na_feature(engine, tmp_path):
    """Missing CB / UB, CB `NA`, UB `nan`, UMIs with N, UMIs of 14-20 bases, mixed UMI lengths in one cell, one UMI in
    several cells, a feature named `NA`: the counts equal the two-step route's."""
    lib, codes = synth.allele_family_library(n_founders=6, alleles_per_founder=1, length=600, snps_mean=0, seed=21)
    lib[1]["columns"][1][0] = "NA"
    lib[1]["columns"][1][1] = "null"
    lib_path = str(tmp_path / "edge.json")
    with open(lib_path, "w") as f:
        json.dump(lib, f)
    reads, truth = synth.sample_reads(codes, 6000, read_len=90, seed=22)
    rng = np.random.default_rng(23)
    cells = ["".join(rng.choice(list("ACGT"), 16)) for _ in range(12)]
    umis = ["".join(rng.choice(list("ACGT"), 10)) for _ in range(40)]
    odd = ["ACGTNACGTN", "NNNNNNNNNN", "ACGTACGTACGTAC", "ACGTACGTACGTACGTACGT", "ACGTACGTACGTACG", "acgtacgt", "AC-GT", "A"]
    recs = []
    for i in range(len(reads)):
        tags = {"CB": cells[i % len(cells)], "UB": umis[rng.integers(0, len(umis))] if i % 5 else odd[i % len(odd)]}
        r = i % 97
        if r == 1:
            del tags["CB"]
        elif r == 2:
            del tags["UB"]
        elif r == 3:
            tags["CB"] = "NA"
        elif r == 4:
            tags["UB"] = "nan"
        elif r == 5:
            tags["CB"] = ""
        recs.append(("e%d" % i, 4, reads[i].tobytes().decode(), tags))
    bam = str(tmp_path / "edge.bam")
    write_bam(bam, recs)
    outs, cnts, o3 = _two_step(engine, tmp_path, lib_path, bam)
    rows = [l.split("\t") for l in open(outs[0]).read().splitlines()[1:]]
    assert any(r[0] == "NA" for r in rows) and any(r[0] == "null" for r in rows)     # the case is exercised
    got = str(tmp_path / "edge_counts.tsv")
    assert frontend.align(lib_path, None, [bam], 2, "unstranded", "", None, engine=engine, counts=got) == 0
    assert o3[0][1] > 10 and _read(got) == _read(cnts[0])
    lg = engine.load_library(lib_path)
    for thr, dis in ((0.2, False), (0.05, True)):
        want = str(tmp_path / "edge_want.tsv")
        x = engine.report_file(outs[0], want, thr, dis)
        assert engine.align_files_counts([bam], [lg], [got], None, thr, dis) == [x] and _read(got) == _read(want)


def test_counts_failure_and_empty_cases(engine, tmp_path, capsys):
    lib, codes = synth.allele_family_library(n_founders=4, alleles_per_founder=2, length=500, snps_mean=4, seed=31)
    lib_path = str(tmp_path / "l.json")
    with open(lib_path, "w") as f:
        json.dump(lib, f)
    # no read is called: empty counts file, rc 0 (write_empty_df)
    rng = np.random.default_rng(32)
    junk = ["".join(rng.choice(list("ACGT"), 80)) for _ in range(300)]
    bam = str(tmp_path / "junk.bam")
    write_bam(bam, [("j%d" % i, 4, s, {"CB": "AAAACCCCGGGGTTTT", "UB": "ACGTACGTAC"}) for i, s in enumerate(junk)])
    got = str(tmp_path / "empty.tsv")
    with open(got, "w") as f:
        f.write("stale")
    assert frontend.align(lib_path, None, [bam], 1, "unstranded", "", None, engine=engine, counts=got) == 0
    assert _read(got) == b"" and "No data to parse" in capsys.readouterr().out
    # FASTQ input: no cell barcodes -> non-zero rc with a message
    fq = tmp_path / "r.fastq"
    fq.write_text("".join("@r%d\n%s\n+\n%s\n" % (i, s, "I" * 80) for i, s in enumerate(junk[:20])))
    assert frontend.align(lib_path, None, [str(fq)], 1, "unstranded", "", None, engine=engine, counts=str(tmp_path / "fq.tsv")) != 0
    assert "FASTQ" in capsys.readouterr().err
    # a BAM without any CB / UB tag
    bare = str(tmp_path / "bare.bam")
    write_bam(bare, [("b%d" % i, 4, s, {}) for i, s in enumerate(junk)])
    assert frontend.align(lib_path, None, [bare], 1, "unstranded", "", None, engine=engine, counts=str(tmp_path / "b.tsv")) != 0
    assert "CB or UB" in capsys.readouterr().err
    # a feature name the per-read TSV cannot carry: NB200_EINVAL naming it (a comma already fails the library load)
    bad = json.loads(json.dumps(lib))
    bad[1]["columns"][1][0] = "HLA-A\r01"
    bad_path = str(tmp_path / "bad.json")
    with open(bad_path, "w") as f:
        json.dump(bad, f)
    lg = engine.load_library(bad_path)
    with pytest.raises(NimbleB200Error) as e:
        engine.align_files_counts([bam], [lg], [str(tmp_path / "x.tsv")])
    assert e.value.code == EINVAL and "HLA-A" in str(e.value)
    bad[1]["columns"][1][0] = "HLA-A,01"
    with open(bad_path, "w") as f:
        json.dump(bad, f)
    assert frontend.align(bad_path, None, [bam], 1, "unstranded", "", None, gpus=[0], counts=str(tmp_path / "y.tsv")) == 1
    assert "HLA-A,01" in capsys.readouterr().err


def test_counts_cross_context(engine, tmp_path):
    """nb200_align_files_counts_multi over two contexts on one GPU ({0, 0}) equals {0} and the two-step route; {0, 1}
    too where the node has two GPUs."""
    import torch
    lib_path, bam = _inputs(tmp_path, 600_000, 41)
    outs, cnts, _ = _two_step(engine, tmp_path, lib_path, bam)
    want = _read(cnts[0])
    assert len(want) > 10_000
    devsets = [[0], [0, 0]] + ([[0, 1]] if torch.cuda.device_count() >= 2 else [])
    for devs in devsets:
        tsv, got = str(tmp_path / "m.tsv"), str(tmp_path / "m_counts.tsv")
        assert frontend.align(lib_path, tsv, [bam], 8, "unstranded", "", None, gpus=devs, counts=got) == 0
        assert _read(got) == want, devs
        assert _read(tsv) == _read(outs[0]), devs
    if len(devsets) < 3:
        pytest.skip("the {0, 1} half needs two GPUs")
