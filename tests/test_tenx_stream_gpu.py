"""The streaming 10x routes: fastq-to-bam (nb200_fastq_to_bam), align --map (nb200_align_10x_fastq(_multi)) and
fastq-to-counts --output.  Records and rows are compared with the oracle's correction over the whole file and with the
two-step route (fastq-to-bam, then align on its BAM)."""
import gzip
import json
import os

import numpy as np
import pytest

from nimble_b200 import frontend, synth
from oracle import oracle as O
from oracle import a5_py as A

pytestmark = pytest.mark.gpu

SLAB = 1 << 17
KEYS = ("total_pairs", "written_pairs", "cb_perfect_match", "cb_corrected", "cb_no_correction", "name_mismatch", "too_short",
        "no_remaining_seq", "cache_size")


def _read(p):
    with open(p, "rb") as f:
        return f.read()


def _write_fastq(path, recs, gz=False):
    text = "".join("@%s\n%s\n+\n%s\n" % r for r in recs)
    with (gzip.open(path, "wb") if gz else open(path, "wb")) as f:
        f.write(text.encode("latin-1"))


def _two_gpus():
    import torch
    return torch.cuda.device_count() >= 2


@pytest.fixture(scope="module")
def tenx(tmp_path_factory):
    """300 k pairs (three slabs) on a clustered whitelist: R1 = CB (errors, N, bytes outside ACGTN, off-whitelist) + UMI +
    62 bases, R2 = 90 bases; every 97th pair has another name in R2, every 101st an R1 too short for CB + UMI, every 103rd
    an R1 of exactly CB + UMI.  Returns the paths, the library and what the oracle needs."""
    tmp = tmp_path_factory.mktemp("tenx")
    lib, codes = synth.allele_family_library(n_founders=8, alleles_per_founder=20, length=700, snps_mean=10, seed=301)
    libp = str(tmp / "lib.json")
    with open(libp, "w") as f:
        json.dump(lib, f)
    n = 300_000
    rng = np.random.default_rng(302)
    r2, _ = synth.sample_reads(codes, n, read_len=90, seed=303)
    tail, _ = synth.sample_reads(codes, n, read_len=62, seed=304)
    wl_a, cb, q = synth.barcode_workload(n, n_whitelist=2000, n_cells=300, err_rate=0.02, n_rate=0.003, off_whitelist=0.02,
                                         seed=305, clustered=0.5)
    junk = rng.random(n) < 0.001
    cb[junk, rng.integers(0, 16, int(junk.sum()))] = np.frombuffer(b"x.a", np.uint8)[rng.integers(0, 3, int(junk.sum()))]
    umi = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, size=(n, 12))]
    q1 = (rng.integers(2, 41, size=(n, 62)) + 33).astype(np.uint8)
    recs1, recs2, el, rows = [], [], np.zeros(n, np.uint8), []
    for i in range(n):
        c, u, t = cb[i].tobytes().decode(), umi[i].tobytes().decode(), tail[i].tobytes().decode()
        qq = "".join(chr(33 + int(x)) for x in q[i]) + "F" * 12 + q1[i].tobytes().decode()
        name2 = "p%d/2" % i
        if i % 97 == 1:
            name2 = "x%d/2" % i
        elif i % 101 == 2:
            c, u, t = c[:10], "", ""
        elif i % 103 == 3:
            t = ""
        else:
            el[i] = 1
        s1 = c + u + t
        recs1.append(("p%d/1" % i, s1, qq[:len(s1)]))
        recs2.append((name2, r2[i].tobytes().decode(), "G" * 90))
        rows.append((u, t, qq[28:len(s1)], r2[i].tobytes().decode()))
    f1, f2 = str(tmp / "R1.fastq.gz"), str(tmp / "R2.fastq")
    _write_fastq(f1, recs1, gz=True)
    _write_fastq(f2, recs2)
    wl_s = [bytes(r).decode() for r in wl_a]
    wlp = str(tmp / "wl.txt")
    with open(wlp, "w") as f:
        f.write("\n".join(wl_s) + "\n")
    return dict(tmp=tmp, libp=libp, f1=f1, f2=f2, wlp=wlp, wl=wl_s, cb=cb, q=q, el=el, rows=rows, n=n)


def test_fastq_to_bam_cross_slab_cache_rule(engine, tenx):
    """Records in order and every counter, cache_size included, equal the oracle's correction over the whole file; the
    oracle over slab-sized chunks disagrees on some reads (a slab-local cache rule would fail)."""
    T = tenx
    o_idx, o_st, o_stats = O.cb_correct(T["wl"], T["cb"], T["q"], T["el"], 16)
    chunk = np.concatenate([O.cb_correct(T["wl"], T["cb"][a:a + SLAB], T["q"][a:a + SLAB], T["el"][a:a + SLAB], 16)[0]
                            for a in range(0, T["n"], SLAB)])
    assert (chunk != o_idx).sum() > 0
    out = str(T["tmp"] / "x.bam")
    st = engine.fastq_to_bam(T["f1"], T["f2"], T["wlp"], out)
    written = np.nonzero((o_st == A.CB_PERFECT) | (o_st == A.CB_CORRECTED))[0]
    want = dict(o_stats, total_pairs=T["n"], written_pairs=len(written), name_mismatch=sum(1 for i in range(T["n"]) if i % 97 == 1),
                too_short=sum(1 for i in range(T["n"]) if i % 97 != 1 and i % 101 == 2),
                no_remaining_seq=sum(1 for i in range(T["n"]) if i % 97 != 1 and i % 101 != 2 and i % 103 == 3))
    for k in KEYS:
        assert st[k] == want[k], k
    assert st["n_multi"] > 0 and st["cb_corrected"] > 1000
    recs = frontend.read_bam(out, with_qual=True)
    assert len(recs) == 2 * len(written)
    for j, i in enumerate(written):
        u, t, qt, s2 = T["rows"][i]
        tags = {"CB": T["wl"][o_idx[i]], "UB": u}
        assert recs[2 * j] == ("p%d" % i, 77, t, tags, -1, qt), i
        assert recs[2 * j + 1] == ("p%d" % i, 141, s2, tags, -1, "G" * 90), i
    assert not os.path.exists(out + ".tmp")


@pytest.mark.parametrize("devs", [[0], [0, 0], pytest.param([0, 1], marks=pytest.mark.skipif(not _two_gpus(), reason="needs two GPUs"))],
                         ids=["0", "0-0", "0-1"])
def test_align_map_contexts_equal_two_steps(engine, tenx, devs):
    """align --map on contexts {0}, {0, 0}, {0, 1} writes the per-read TSV of fastq-to-bam followed by align, byte for byte;
    a .gz output decompresses to the same text."""
    T = tenx
    want = str(T["tmp"] / "two_step.tsv")
    if "bam_stats" not in T:
        bam = str(T["tmp"] / "two.bam")
        T["bam_stats"] = engine.fastq_to_bam(T["f1"], T["f2"], T["wlp"], bam)
        engine.align_files([bam], [engine.load_library(T["libp"])], [want])
    text = _read(want)
    assert text.count(b"\n") > 100_000
    tag = "_".join(map(str, devs))
    got = str(T["tmp"] / ("map_%s.tsv" % tag))
    assert frontend.align_10x(T["libp"], got, T["f1"], T["f2"], T["wlp"], 8, gpus=devs) == 0
    assert _read(got) == text
    gz = got + ".gz"
    assert frontend.align_10x(T["libp"], gz, T["f1"], T["f2"], T["wlp"], 8, gpus=devs) == 0
    with gzip.open(gz, "rb") as g:
        assert g.read() == text
    if devs == [0]:                                   # the one-context entry (Engine.align_10x_fastq)
        one = str(T["tmp"] / "one.tsv")
        st = engine.align_10x_fastq(T["f1"], T["f2"], T["wlp"], [engine.load_library(T["libp"])], [one])
        assert _read(one) == text
    else:                                             # the multi entry: hit flags or-ed and miss logs gathered across contexts
        one = str(T["tmp"] / ("multi_%s.tsv" % tag))
        st, _ = frontend._align_10x_multi(devs, 8, T["f1"], T["f2"], T["wlp"], [T["libp"]], "unstranded", None, "", 16, 12, [one])
        assert _read(one) == text
    for k in KEYS:
        assert st[k] == T["bam_stats"][k], k
    assert st["cache_size"] > 1000


def test_fastq_to_counts_output(engine, tenx, capsys):
    """fastq-to-counts --output: the counts files are those of a run without --output, the per-read TSV that of align --map."""
    T = tenx
    plain = str(T["tmp"] / "counts_plain.tsv")
    assert frontend.fastq_to_counts(T["libp"], T["f1"], T["f2"], T["wlp"], plain, 8, engine=engine) == 0
    cnt, per_read = str(T["tmp"] / "counts_out.tsv"), str(T["tmp"] / "per_read.tsv")
    assert frontend.fastq_to_counts(T["libp"], T["f1"], T["f2"], T["wlp"], cnt, 8, output=per_read) == 0
    assert _read(cnt) == _read(plain) and len(_read(cnt)) > 1000
    mapped = str(T["tmp"] / "map_for_counts.tsv")
    assert frontend.align_10x(T["libp"], mapped, T["f1"], T["f2"], T["wlp"], 8, engine=engine) == 0
    assert _read(per_read) == _read(mapped)
    assert "wrote %s" % per_read in capsys.readouterr().out


def _small(tmp_path, codes, extra, name="s"):
    """400 corrected pairs around one extra pair (name, R1, R2); returns R1 / R2 paths."""
    r2, _ = synth.sample_reads(codes, 400, read_len=90, seed=311)
    tail, _ = synth.sample_reads(codes, 400, read_len=60, seed=312)
    good = [("g%d" % i, "ACGTACGTACGTACGT" + "".join("ACGT"[(i >> (2 * k)) & 3] for k in range(12)) + tail[i].tobytes().decode(),
             r2[i].tobytes().decode()) for i in range(400)]
    recs = good[:200] + [extra] + good[200:]
    f1, f2 = str(tmp_path / ("%s_1.fastq" % name)), str(tmp_path / ("%s_2.fastq" % name))
    _write_fastq(f1, [(n, a, "F" * len(a)) for n, a, _ in recs])
    _write_fastq(f2, [(n, b, "F" * len(b)) for n, _, b in recs])
    return f1, f2


def test_over_long_reads_and_names(engine, tmp_path):
    """fastq-to-bam writes a corrected pair whose reads exceed 500 bases; a corrected pair with a name over 254 bytes fails,
    and so does align --map on a corrected pair over 500 bases.  Without a correction the same pairs pass."""
    lib, codes = synth.allele_family_library(n_founders=4, alleles_per_founder=6, length=700, snps_mean=6, seed=313)
    libp = str(tmp_path / "lib.json")
    with open(libp, "w") as f:
        json.dump(lib, f)
    lg = engine.load_library(libp)
    wlp = str(tmp_path / "wl.txt")
    with open(wlp, "w") as f:
        f.write("ACGTACGTACGTACGT\nTTTTTTTTTTTTTTTT\n")
    umi = "ACGTTGCAACGT"
    for cb, corrected in (("ACGTACGTACGTACGA", True), ("GGGGGGGGGGGGGGGG", False)):
        f1, f2 = _small(tmp_path, codes, ("long", cb + umi + "A" * 520, "C" * 530), "r%d" % corrected)
        out = str(tmp_path / "long.bam")
        st = engine.fastq_to_bam(f1, f2, wlp, out)
        recs = frontend.read_bam(out)
        assert st["written_pairs"] == 400 + corrected and len(recs) == 2 * (400 + corrected)
        if corrected:
            assert recs[400][0] == "long" and recs[400][2] == "A" * 520 and recs[401][2] == "C" * 530
        tsv = str(tmp_path / "long.tsv")
        if corrected:
            with pytest.raises(Exception) as e:
                engine.align_10x_fastq(f1, f2, wlp, [lg], [tsv])
            assert "500 bases" in str(e.value) and not os.path.exists(tsv) and not os.path.exists(tsv + ".tmp")
        else:
            engine.align_10x_fastq(f1, f2, wlp, [lg], [tsv])
            engine.align_files([out], [lg], [str(tmp_path / "long_two.tsv")])
            assert _read(tsv) == _read(str(tmp_path / "long_two.tsv"))
        f1, f2 = _small(tmp_path, codes, ("n" * 300, cb + umi + "ACGT" * 10, "C" * 90), "n%d" % corrected)
        out = str(tmp_path / "name.bam")
        if corrected:
            with pytest.raises(Exception) as e:
                engine.fastq_to_bam(f1, f2, wlp, out)
            assert "254 bytes" in str(e.value) and not os.path.exists(out) and not os.path.exists(out + ".tmp")
        else:
            assert engine.fastq_to_bam(f1, f2, wlp, out)["written_pairs"] == 400


def test_failure_after_first_slab_and_empty_input(engine, tenx, tmp_path):
    """A malformed record after the first slab, or in the tail of the longer file, fails the call: no output and no .tmp
    are left and a previous output is intact.  Empty inputs give a header-only BAM and a header-only TSV."""
    T = tenx
    lg = engine.load_library(T["libp"])
    with gzip.open(T["f1"], "rt") as f:
        lines = f.read().split("\n")
    r2 = open(T["f2"]).read().split("\n")
    bad_mid = list(lines)
    bad_mid[4 * 200_000 + 3] = bad_mid[4 * 200_000 + 3][:-1]                # quality shorter than the sequence
    bad_tail = r2[:-1] + ["@extra", "ACGT", "+", "FF", ""]                   # R2 longer than R1, its extra record malformed
    cases = [("mid", "\n".join(bad_mid), "\n".join(r2)), ("tail", "\n".join(lines), "\n".join(bad_tail))]
    for tag, a, b in cases:
        f1, f2 = str(tmp_path / ("%s_1.fastq" % tag)), str(tmp_path / ("%s_2.fastq" % tag))
        open(f1, "w").write(a)
        open(f2, "w").write(b)
        bam, tsv = str(tmp_path / "prev.bam"), str(tmp_path / "prev.tsv")
        open(bam, "wb").write(b"previous bam")
        open(tsv, "w").write("previous tsv")
        with pytest.raises(Exception):
            engine.fastq_to_bam(f1, f2, T["wlp"], bam)
        with pytest.raises(Exception):
            engine.align_10x_fastq(f1, f2, T["wlp"], [lg], [tsv])
        assert frontend.align_10x(T["libp"], tsv, f1, f2, T["wlp"], 4, gpus=[0, 0]) == 1
        assert _read(bam) == b"previous bam" and _read(tsv) == b"previous tsv", tag
        assert not os.path.exists(bam + ".tmp") and not os.path.exists(tsv + ".tmp"), tag
    e1, e2 = str(tmp_path / "e1.fastq"), str(tmp_path / "e2.fastq")
    open(e1, "w").close(); open(e2, "w").close()
    out = str(tmp_path / "empty.bam")
    st = engine.fastq_to_bam(e1, e2, T["wlp"], out)
    assert st["total_pairs"] == 0 and st["cache_size"] == 0 and frontend.read_bam(out) == []
    tsv = str(tmp_path / "empty.tsv")
    engine.align_10x_fastq(e1, e2, T["wlp"], [lg], [tsv])
    assert _read(tsv).decode() == "\t".join(frontend.PER_READ_COLUMNS) + "\n"


def test_long_and_non_acgtn_umis(engine, tmp_path):
    """UMIs of 14 bases and UMIs holding bytes outside ACGTN reach the BAM and the per-read TSV as raw text: fastq-to-bam's
    records, and align --map (one context and the multi entry on {0, 0}) equal fastq-to-bam followed by align."""
    lib, codes = synth.allele_family_library(n_founders=4, alleles_per_founder=6, length=700, snps_mean=6, seed=321)
    libp = str(tmp_path / "lib.json")
    with open(libp, "w") as f:
        json.dump(lib, f)
    lg = engine.load_library(libp)
    wl = ["ACGTACGTACGTACGT", "TTTTTTTTTTTTTTTT", "GATTACAGATTACAGA"]
    wlp = str(tmp_path / "wl.txt")
    with open(wlp, "w") as f:
        f.write("\n".join(wl) + "\n")
    rng = np.random.default_rng(322)
    n = 3000
    r2, _ = synth.sample_reads(codes, n, read_len=90, seed=323)
    tail, _ = synth.sample_reads(codes, n, read_len=60, seed=324)
    cbs = wl + ["ACGTACGTACGTACGA", "GGGGGGGGGGGGGGGG"]                # + a corrected and an uncorrected barcode
    for U in (14, 12):
        recs1, recs2, umis = [], [], []
        for i in range(n):
            u = "".join(rng.choice(list("ACGT"), U))
            if i % 3 == 0:                                              # a byte outside ACGTN: '.', lower case, 'X'
                j = int(rng.integers(0, U))
                u = u[:j] + ".nX"[i % 9 // 3] + u[j + 1:]
            s1 = cbs[i % len(cbs)] + u + tail[i].tobytes().decode()
            recs1.append(("q%d/1" % i, s1, "F" * len(s1)))
            recs2.append(("q%d/2" % i, r2[i].tobytes().decode(), "F" * 90))
            umis.append(u)
        f1, f2 = str(tmp_path / ("u%d_1.fastq" % U)), str(tmp_path / ("u%d_2.fastq" % U))
        _write_fastq(f1, recs1)
        _write_fastq(f2, recs2)
        bam = str(tmp_path / ("u%d.bam" % U))
        st = engine.fastq_to_bam(f1, f2, wlp, bam, 16, U)
        written = [i for i in range(n) if i % len(cbs) != 4]
        assert st["written_pairs"] == len(written) and st["cb_corrected"] > 0
        recs = frontend.read_bam(bam)
        assert len(recs) == 2 * len(written)
        for j, i in enumerate(written):
            assert recs[2 * j][0] == "q%d" % i and recs[2 * j][3] == {"CB": wl[i % len(cbs) % 3 if i % len(cbs) != 3 else 0], "UB": umis[i]}
        want = str(tmp_path / ("u%d_two.tsv" % U))
        engine.align_files([bam], [lg], [want])
        text = _read(want)
        assert text.count(b"\n") > 1000
        one = str(tmp_path / ("u%d_one.tsv" % U))
        st1 = engine.align_10x_fastq(f1, f2, wlp, [lg], [one], 16, U)
        assert _read(one) == text
        multi = str(tmp_path / ("u%d_multi.tsv" % U))
        st2, _ = frontend._align_10x_multi([0, 0], 4, f1, f2, wlp, [libp], "unstranded", None, "", 16, U, [multi])
        assert _read(multi) == text
        for k in KEYS:
            assert st1[k] == st[k] and st2[k] == st[k], k
