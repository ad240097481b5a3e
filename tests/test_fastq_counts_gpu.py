"""`fastq-to-counts` (nb200_fastq_to_counts / nb200_fastq_to_counts_multi): raw 10x R1 / R2 FASTQ to the counts TSV in one
streaming pass.  Every case compares the counts file byte for byte, out3 and fastq-to-bam's counters with the two-step
route: fastq-to-bam, then align --counts on its BAM."""
import gzip
import json

import numpy as np
import pytest

from nimble_b200 import frontend, synth
from nimble_b200.__main__ import main
from oracle import oracle as O

pytestmark = pytest.mark.gpu

KEYS = ("total_pairs", "written_pairs", "cb_perfect_match", "cb_corrected", "cb_no_correction", "name_mismatch", "too_short",
        "no_remaining_seq")
SLAB = 1 << 17


def _read(p):
    with open(p, "rb") as f:
        return f.read()


def _write_fastq(path, recs, gz=False, eol="\n", final_eol=True):
    text = eol.join("@%s%s%s%s+%s%s" % (n, eol, s, eol, eol, q) for n, s, q in recs)
    if recs and final_eol:
        text += eol
    with (gzip.open(path, "wb") if gz else open(path, "wb")) as f:
        f.write(text.encode("latin-1"))


def _library(tmp_path, seed, name="lib", prefix=None):
    kw = {"name_prefix": prefix} if prefix else {}
    lib, codes = synth.allele_family_library(n_founders=8, alleles_per_founder=20, length=700, snps_mean=10, seed=seed, **kw)
    p = str(tmp_path / ("%s.json" % name))
    with open(p, "w") as f:
        json.dump(lib, f)
    return p, codes


def _tenx(tmp_path, codes, n, seed, clustered=0.5, gz1=False, tag="in"):
    """n pairs: R1 = CB (16, synth.barcode_workload with errors, N and off-whitelist barcodes) + UMI (12) + 62 bases, R2 = 90
    bases, random qualities; returns (R1 path, R2 path, whitelist path, whitelist, cb, cb phred)."""
    rng = np.random.default_rng(seed)
    r2, _ = synth.sample_reads(codes, n, read_len=90, seed=seed + 1)
    tail, _ = synth.sample_reads(codes, n, read_len=62, seed=seed + 2)
    wl_a, cb, q = synth.barcode_workload(n, n_whitelist=2000, n_cells=300, err_rate=0.02, n_rate=0.002, off_whitelist=0.02,
                                         seed=seed + 3, clustered=clustered)
    pool = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, size=(1500, 12))]
    umi = pool[rng.integers(0, len(pool), size=n)]
    q1 = (rng.integers(2, 41, size=(n, 74)) + 33).astype(np.uint8)
    q2 = (rng.integers(2, 41, size=(n, 90)) + 33).astype(np.uint8)
    s1 = np.concatenate([cb, umi, tail], axis=1)
    qq1 = np.concatenate([(q + 33).astype(np.uint8), q1], axis=1)
    f1, f2 = str(tmp_path / ("%s_R1.fastq%s" % (tag, ".gz" if gz1 else ""))), str(tmp_path / ("%s_R2.fastq" % tag))
    _write_fastq(f1, [("p%d/1" % i, s1[i].tobytes().decode(), qq1[i].tobytes().decode()) for i in range(n)], gz=gz1)
    _write_fastq(f2, [("p%d/2" % i, r2[i].tobytes().decode(), q2[i].tobytes().decode()) for i in range(n)])
    wl_s = [bytes(r).decode() for r in wl_a]
    wlp = str(tmp_path / ("%s_wl.txt" % tag))
    with open(wlp, "w") as f:
        f.write("\n".join(wl_s) + "\n")
    return f1, f2, wlp, wl_s, cb, q


def _check(engine, tmp_path, f1, f2, wlp, libs, cb_len=16, umi_len=12, thr=0.05, dis=False, tag="x"):
    """fastq_to_counts equals fastq_to_bam -> align_files_counts: bytes of every counts file, out3, the counters."""
    bam = str(tmp_path / ("%s.bam" % tag))
    st_a = engine.fastq_to_bam(f1, f2, wlp, bam, cb_len, umi_len)
    want = [str(tmp_path / ("%s.want.%d.tsv" % (tag, i))) for i in range(len(libs))]
    o3_a = engine.align_files_counts([bam], libs, want, None, thr, dis)
    got = [str(tmp_path / ("%s.got.%d.tsv" % (tag, i))) for i in range(len(libs))]
    st_b, o3_b = engine.fastq_to_counts(f1, f2, wlp, libs, got, cb_len, umi_len, thr, dis)
    assert o3_b == o3_a, tag
    for w, g in zip(want, got):
        assert _read(g) == _read(w), tag
    for k in KEYS:
        assert st_b[k] == st_a[k], (tag, k)
    assert st_b["cache_size"] == 0
    return st_a, o3_a, [_read(w) for w in want]


def test_three_slabs_thresholds_and_cross_slab_cache_rule(engine, tmp_path):
    """300 k pairs (three slabs) on a clustered whitelist at thresholds 0.05, 0.2 and none.  The oracle over the whole file and
    over 2^17-pair chunks disagree on some reads: a slab-local cache rule would fail the comparison."""
    lib_path, codes = _library(tmp_path, 91)
    n = 300_000
    f1, f2, wlp, wl_s, cb, q = _tenx(tmp_path, codes, n, 92)
    o_all, _, _ = O.cb_correct(wl_s, cb, q, None, 16)
    o_chunk = np.concatenate([O.cb_correct(wl_s, cb[a:a + SLAB], q[a:a + SLAB], None, 16)[0] for a in range(0, n, SLAB)])
    assert (o_all != o_chunk).sum() > 0
    lib = engine.load_library(lib_path)
    for thr, dis in ((0.05, False), (0.2, False), (0.05, True)):
        st, o3, _ = _check(engine, tmp_path, f1, f2, wlp, [lib], thr=thr, dis=dis, tag="t%s%d" % (thr, dis))
        assert st["n_multi"] > 0 and o3[0][0] > 100_000 and o3[0][1] > 1000
    assert st["total_pairs"] == n and st["cb_corrected"] > 1000


def test_two_libraries_trim_gzip_r1(engine, tmp_path):
    """Two libraries with --trim "70:0.6,90:0.4", R1 gzip-compressed and R2 plain; the front end names the files as align."""
    pa, codes = _library(tmp_path, 11, "liba")
    pb, _ = _library(tmp_path, 11, "libb", prefix="Mafa")
    f1, f2, wlp, _, _, _ = _tenx(tmp_path, codes, 40_000, 12, clustered=0.3, gz1=True)
    libs = [engine.load_library(pa), engine.load_library(pb)]
    for lg, (t, s) in zip(libs, ((70, 0.6), (90, 0.4))):
        lg.set_trim(t, s)
    _, o3, want = _check(engine, tmp_path, f1, f2, wlp, libs, tag="trim")
    assert all(x[0] > 10_000 for x in o3)
    cnt = str(tmp_path / "fe_counts.tsv")
    assert frontend.fastq_to_counts("%s,%s" % (pa, pb), f1, f2, wlp, cnt, 4, trim="70:0.6,90:0.4", engine=engine) == 0
    got = frontend._per_library_paths(cnt, [pa, pb])
    assert got == [str(tmp_path / "fe_counts.liba.tsv"), str(tmp_path / "fe_counts.libb.tsv")]
    assert [_read(g) for g in got] == want


def test_edge_input(engine, tmp_path):
    """CRLF, no final newline, R2 longer than R1, lower-case bases, /1 /2 suffixes, a name mismatch, too short, no remaining
    sequence, N and junk bytes in the CB, off-whitelist barcodes, several candidates with other qualities, R1 over 500 bases;
    then NA-token UMIs, a whitelist holding `NA` with --cb-length 2, and --umi-length 0."""
    lib_path, codes = _library(tmp_path, 21)
    lib = engine.load_library(lib_path)
    rng = np.random.default_rng(22)
    n = 3000
    r2, _ = synth.sample_reads(codes, n, read_len=90, seed=23)
    tail, _ = synth.sample_reads(codes, n, read_len=60, seed=24)
    longt, _ = synth.sample_reads(codes, 20, read_len=480, seed=25)
    wl = ["ACGTACGTACGTACGT", "TTTTTTTTTTTTTTTT", "AAAAAAAAAAAAAAAC", "AAAAAAAAAAAAAACA", "GATTACAGATTACAGA"]
    cbs = wl + ["ACGTACGTNCGTACGT", "ACGTACGT.CGTACGT", "GGGGGGGGGGGGGGGG", "AAAAAAAAAAAAAAAA", "GATTACAGATTACAGT", "acgtACGTACGTACGT"]
    umis = ["".join(rng.choice(list("ACGT"), 12)) for _ in range(n)]     # (few reads per UMI: intersections stay non-empty)
    rec1, rec2 = [], []
    for i in range(n):
        cb = cbs[i % len(cbs)]
        q = "".join(chr(33 + int(x)) for x in rng.integers(2, 41, 16))
        t = tail[i].tobytes().decode()
        kind = i % 13
        name1, name2 = "r%d/1" % i, "r%d/2" % i
        if kind == 1:
            t = t.lower()
        elif kind == 2:
            name2 = "s%d/2" % i                                  # name mismatch
        elif kind == 3:
            t, cb = "", cb[:8]                                    # too short
        elif kind == 4:
            t = ""                                                # no remaining sequence
        elif kind == 5 and i < 13 * 20:
            t = longt[i // 13].tobytes().decode()                 # R1 of 508 bases
        elif kind == 6:
            name1, name2 = "r%d" % i, "r%d" % i
        s1 = cb + umis[i % len(umis)] + t
        rec1.append((name1 + " extra", s1, q[:len(cb)] + "F" * (len(s1) - len(cb))))
        rec2.append((name2, r2[i].tobytes().decode(), "F" * 90))
    rec2 += [("z%d" % j, "ACGT", "FFFF") for j in range(5)]          # R2 longer than R1: zip stops at the shorter file
    f1, f2, wlp = str(tmp_path / "e1.fastq"), str(tmp_path / "e2.fastq"), str(tmp_path / "ewl.txt")
    _write_fastq(f1, rec1, eol="\r\n", final_eol=False)
    _write_fastq(f2, rec2)
    with open(wlp, "w") as f:
        f.write("\n".join(wl) + "\n")
    st, o3, _ = _check(engine, tmp_path, f1, f2, wlp, [lib], tag="edge")
    assert st["name_mismatch"] > 0 and st["too_short"] > 0 and st["no_remaining_seq"] > 0 and st["cb_corrected"] > 0
    assert st["cb_no_correction"] > 0 and o3[0][1] > 10

    # NA-token UMIs: --umi-length 2 and 4 (report drops such rows)
    for U, tokens in ((2, ["NA", "AC", "GT", "TT"]), (4, ["NULL", "None", "ACGT", "-nan", "TTAA", "GGCC"])):
        r1 = [(n_, wl[i % 2] + tokens[i % len(tokens)] + tail[i].tobytes().decode(), "F" * (16 + U + 60)) for i, n_ in
              enumerate("u%d" % j for j in range(n))]
        g1, g2 = str(tmp_path / ("u%d_1.fastq" % U)), str(tmp_path / ("u%d_2.fastq" % U))
        _write_fastq(g1, r1)
        _write_fastq(g2, [("u%d" % i, r2[i].tobytes().decode(), "F" * 90) for i in range(n)])
        _, o3, _ = _check(engine, tmp_path, g1, g2, wlp, [lib], umi_len=U, tag="umi%d" % U)
        assert o3[0][0] > 0

    # a whitelist holding NA, --cb-length 2: reads corrected to NA (exactly, or as a candidate) are not counted
    wl2 = str(tmp_path / "wl2.txt")
    with open(wl2, "w") as f:
        f.write("NA\nAC\nGT\nCC\n")
    cb2 = ["NA", "AC", "NC", "GG", "GT", "TC"]
    r1 = [("c%d" % i, cb2[i % len(cb2)] + umis[i][:4] + tail[i].tobytes().decode(),
           "".join(chr(33 + int(x)) for x in rng.integers(2, 41, 2)) + "F" * 64) for i in range(n)]
    g1, g2 = str(tmp_path / "c1.fastq"), str(tmp_path / "c2.fastq")
    _write_fastq(g1, r1)
    _write_fastq(g2, [("c%d" % i, r2[i].tobytes().decode(), "F" * 90) for i in range(n)])
    st, o3, want = _check(engine, tmp_path, g1, g2, wl2, [lib], cb_len=2, umi_len=4, tag="cbna")
    assert st["n_multi"] > 0 and o3[0][0] > 0 and b"\tNA\n" not in want[0]

    # --umi-length 0: every UB is empty, every row is dropped
    _, o3, want = _check(engine, tmp_path, f1, f2, wlp, [lib], umi_len=0, tag="umi0")
    assert o3[0] == (0, 0, 0) and want == [b""]


def test_failures_and_empty_input(engine, tmp_path, capsys):
    lib_path, codes = _library(tmp_path, 31)
    wlp = str(tmp_path / "wl.txt")
    with open(wlp, "w") as f:
        f.write("ACGTACGTACGTACGT\nTTTTTTTTTTTTTTTT\n")
    cnt = str(tmp_path / "c.tsv")
    # empty FASTQs: empty counts file, rc 0
    e1, e2 = str(tmp_path / "e1.fastq"), str(tmp_path / "e2.fastq")
    open(e1, "w").close(); open(e2, "w").close()
    with open(cnt, "w") as f:
        f.write("stale")
    assert frontend.fastq_to_counts(lib_path, e1, e2, wlp, cnt, engine=engine) == 0
    assert _read(cnt) == b"" and "No data to parse" in capsys.readouterr().out
    # standard 28-base 10x R1: every pair is dropped (no_remaining_seq), empty file, rc 0, a note on stderr
    r2, _ = synth.sample_reads(codes, 500, read_len=90, seed=32)
    _write_fastq(e1, [("p%d" % i, "ACGTACGTACGTACGT" + "ACGTACGTACGT", "F" * 28) for i in range(500)])
    _write_fastq(e2, [("p%d" % i, r2[i].tobytes().decode(), "F" * 90) for i in range(500)])
    assert frontend.fastq_to_counts(lib_path, e1, e2, wlp, cnt, engine=engine) == 0
    out = capsys.readouterr()
    assert _read(cnt) == b"" and "No remaining sequence: 500" in out.out and "no read 1 is left" in out.err
    # a missing file, a sequence / quality length mismatch: rc != 0 with a message
    assert frontend.fastq_to_counts(lib_path, str(tmp_path / "nope.fastq"), e2, wlp, cnt, engine=engine) != 0
    assert "nope.fastq" in capsys.readouterr().err
    _write_fastq(e1, [("p0", "ACGTACGTACGTACGT" + "ACGTACGTACGT" + "ACGT", "F" * 30)])
    assert frontend.fastq_to_counts(lib_path, e1, e2, wlp, cnt, engine=engine) != 0
    assert "quality lengths differ" in capsys.readouterr().err


def _two_gpus():
    import torch
    return torch.cuda.device_count() >= 2


@pytest.fixture(scope="module")
def big_input(engine, tmp_path_factory):
    """600 k pairs and the two-step route's counts on them (shared by the device sets below)."""
    tmp_path = tmp_path_factory.mktemp("ctx")
    lib_path, codes = _library(tmp_path, 41)
    f1, f2, wlp, _, _, _ = _tenx(tmp_path, codes, 600_000, 42)
    _, o3, want = _check(engine, tmp_path, f1, f2, wlp, [engine.load_library(lib_path)], tag="one")
    assert o3[0][0] > 200_000
    return tmp_path, lib_path, f1, f2, wlp, want[0]


@pytest.mark.parametrize("devs", [[0], [0, 0], pytest.param([0, 1], marks=pytest.mark.skipif(not _two_gpus(), reason="needs two GPUs"))],
                         ids=["0", "0-0", "0-1"])
def test_contexts_give_identical_bytes(big_input, devs):
    """Contexts {0}, {0, 0} and {0, 1} (where the node has two GPUs) on 600 k pairs write the two-step route's bytes."""
    tmp_path, lib_path, f1, f2, wlp, want = big_input
    got = str(tmp_path / ("m_counts_%s.tsv" % "_".join(map(str, devs))))
    assert frontend.fastq_to_counts(lib_path, f1, f2, wlp, got, 8, gpus=devs) == 0
    assert _read(got) == want


def test_over_long_pairs_fail_only_when_written(engine, tmp_path):
    """A pair with R1 over 500 bases after the cut, R2 over 500 bases or a name over 254 bytes: the two steps drop it without
    failing when its barcode gets no correction, and fail when it is corrected (fastq-to-bam writes it).  So does this route,
    and the pair's barcode still takes part in the correction."""
    lib_path, codes = _library(tmp_path, 61)
    lib = engine.load_library(lib_path)
    r2, _ = synth.sample_reads(codes, 400, read_len=90, seed=62)
    tail, _ = synth.sample_reads(codes, 400, read_len=60, seed=63)
    wlp = str(tmp_path / "wl.txt")
    with open(wlp, "w") as f:
        f.write("ACGTACGTACGTACGT\nTTTTTTTTTTTTTTTT\n")
    umi = "ACGTTGCAACGT"
    good = [("g%d" % i, "ACGTACGTACGTACGT" + "".join("ACGT"[(i >> (2 * k)) & 3] for k in range(12)) + tail[i].tobytes().decode(),
             r2[i].tobytes().decode()) for i in range(400)]                       # (one read per UMI)
    bad = {"r1": ("long_r1", "GGGGGGGGGGGGGGGG" + umi + "A" * 501, "C" * 90),
           "r2": ("long_r2", "GGGGGGGGGGGGGGGG" + umi + "ACGT" * 10, "C" * 501),
           "name": ("n" * 300, "GGGGGGGGGGGGGGGG" + umi + "ACGT" * 10, "C" * 90)}
    for kind, (nm, s1, s2) in bad.items():
        for cb, fails in (("GGGGGGGGGGGGGGGG", False), ("ACGTACGTACGTACGT", True)):    # off-whitelist / a perfect match
            recs = good[:200] + [(nm, cb + s1[16:], s2)] + good[200:]
            f1, f2 = str(tmp_path / ("%s_1.fastq" % kind)), str(tmp_path / ("%s_2.fastq" % kind))
            _write_fastq(f1, [(n_, a, "F" * len(a)) for n_, a, _ in recs])
            _write_fastq(f2, [(n_, b, "F" * len(b)) for n_, _, b in recs])
            if not fails:
                st, o3, _ = _check(engine, tmp_path, f1, f2, wlp, [lib], tag="%s_ok" % kind)
                assert st["cb_no_correction"] == 1 and st["written_pairs"] == 400 and o3[0][0] > 0
                continue
            with pytest.raises(Exception):
                bam = str(tmp_path / "b.bam")
                engine.fastq_to_bam(f1, f2, wlp, bam)                                   # (a name over 254 bytes fails here)
                engine.align_files_counts([bam], [lib], [str(tmp_path / "b.tsv")])      # (an over-long read here)
            with pytest.raises(Exception) as e:
                engine.fastq_to_counts(f1, f2, wlp, [lib], [str(tmp_path / "c.tsv")])
            assert ("254 bytes" if kind == "name" else "500 bases") in str(e.value)


def test_fastq_to_bam_front_end_unchanged(engine, tmp_path, capsys):
    """fastq-to-bam's front end still ends with the output line and returns the statistics."""
    lib_path, codes = _library(tmp_path, 71)
    f1, f2, wlp, _, _, _ = _tenx(tmp_path, codes, 2000, 72, clustered=0.3)
    out = str(tmp_path / "o.bam")
    st = frontend.fastq_to_bam_with_barcodes(f1, f2, wlp, out, 2, engine=engine)
    text = capsys.readouterr().out
    assert st["total_pairs"] == 2000 and st["written_pairs"] > 1000
    assert "Correction cache size: %d unique raw CBs" % st["cache_size"] in text
    assert text.rstrip().endswith("Output BAM written to: %s" % out)


def test_cli_end_to_end(engine, tmp_path, capsys):
    lib_path, codes = _library(tmp_path, 51)
    f1, f2, wlp, _, _, _ = _tenx(tmp_path, codes, 20_000, 52, clustered=0.3)
    _, _, want = _check(engine, tmp_path, f1, f2, wlp, [engine.load_library(lib_path)], tag="cli")
    got = str(tmp_path / "cli_counts.tsv")
    capsys.readouterr()
    with pytest.raises(SystemExit) as e:
        main(["fastq-to-counts", "--reference", lib_path, "--r1-fastq", f1, "--r2-fastq", f2, "--map", wlp, "--counts", got, "-c", "4"])
    assert e.value.code == 0 and _read(got) == want[0]
    out = capsys.readouterr().out
    assert "Total read pairs: 20000" in out and "Dropped " in out
