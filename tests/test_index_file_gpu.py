"""Loading a library from an index file (`index`, then --reference LIB.nb200idx) against building it from the JSON:
every route that takes a library path gives the same bytes, and a damaged image is refused on the device."""
import json
import os
import subprocess

import numpy as np
import pytest

from nimble_b200 import frontend, synth
from nimble_b200._lib import EINVAL, NimbleB200Error
from test_fastq_counts_gpu import _tenx
from test_frontend import write_bam

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ALIGNER = os.path.join(ROOT, "nimble_b200", "aligner")


def _read(p):
    with open(p, "rb") as f:
        return f.read()


def _dump(obj, path):
    with open(path, "w") as f:
        json.dump(obj, f)
    return str(path)


def _index(json_path, out, k, monkeypatch, lf=None):
    """Index file of json_path at k; with lf the table is built dense (NB200_TABLE_LF at write time only)."""
    if lf:
        monkeypatch.setenv("NB200_TABLE_LF", lf)
    assert frontend.index(json_path, str(out), k=k, num_cores=8) == 0
    monkeypatch.delenv("NB200_TABLE_LF", raising=False)
    return str(out)


SHAPES = {
    # allele family at k = 20, default (sparse) table
    "allele_k20": (lambda: synth.allele_family_library(n_founders=8, alleles_per_founder=20, length=700, snps_mean=10, seed=61), 20, None),
    # transcripts at k = 31 with a dense table
    "transcript_k31_dense": (lambda: synth.random_transcript_library(n_seqs=400, mean_len=1500, family_frac=0.4, seed=62), 31, "0.9"),
}


@pytest.fixture(params=sorted(SHAPES))
def shape(request, tmp_path, monkeypatch):
    make, k, lf = SHAPES[request.param]
    lib, codes = make()
    js = _dump(lib, tmp_path / "lib.json")
    idx = _index(js, tmp_path / "lib.nb200idx", k, monkeypatch, lf)
    return js, idx, codes, k, lf


def _json_lib(engine, js, k, lf, monkeypatch, **kw):
    if lf:
        monkeypatch.setenv("NB200_TABLE_LF", lf)
    try:
        return engine.load_library(js, k=k, **kw)
    finally:
        monkeypatch.delenv("NB200_TABLE_LF", raising=False)


def test_resident_align_index_equals_json(engine, shape, monkeypatch):
    js, idx, codes, k, lf = shape
    a = _json_lib(engine, js, k, lf, monkeypatch)
    b = engine.load_library(idx)                                  # k: the index's own
    assert b.info == a.info and bytes(b.config) == bytes(a.config) and b.feature_names == a.feature_names
    r1, truth = synth.sample_reads(codes, 60_000, read_len=100, seed=k)
    key = synth.barcodes_10x(len(r1), n_cells=200, seed=k, truth=truth)
    ta, ra, fa = engine.align(a, r1, key=key, per_read=True)
    tb, rb, fb = engine.align(b, r1, key=key, per_read=True)
    assert ra.tobytes() == rb.tobytes() and np.array_equal(fa, fb)
    assert (ra["reason"] == 0).sum() > 30_000
    for f in ("cell", "count", "feat_off", "feat_ids"):
        assert np.array_equal(getattr(ta, f), getattr(tb, f)), f
    assert ta.dropped_empty == tb.dropped_empty
    # strand filter and config setters act on an index library as on a JSON one
    c = engine.load_library(idx, strand_filter="fiveprime", k=k)
    d = _json_lib(engine, js, k, lf, monkeypatch, strand_filter="fiveprime")
    assert bytes(c.config) == bytes(d.config) and c.config.strand_filter == 1
    assert engine.align(c, r1, per_read=True)[1].tobytes() == engine.align(d, r1, per_read=True)[1].tobytes()


def _pairs_bam(tmp_path, codes, n, seed):
    m1, m2, truth = synth.sample_pairs(codes, n, read_len=120, seed=seed)
    key = synth.barcodes_10x(n, n_cells=80, seed=seed + 1, truth=truth)
    rng = np.random.default_rng(seed + 2)
    q1, q2 = rng.integers(2, 41, size=m1.shape), rng.integers(2, 41, size=m2.shape)
    recs = []
    for i in range(n):
        tags = {"CB": synth.unpack_barcode(int(key[i]) >> 32, 16), "UB": synth.unpack_barcode(int(key[i]) & 0xFFFFFF, 12)}
        recs.append(("p%d" % i, 77, m1[i].tobytes().decode(), tags, q1[i]))
        recs.append(("p%d" % i, 141, m2[i].tobytes().decode(), tags, q2[i]))
    bam = str(tmp_path / "pairs.bam")
    write_bam(bam, recs)
    return bam


@pytest.fixture(scope="module")
def two_libs(tmp_path_factory):
    """An allele library (JSON, k = 20) and a transcript library (index at k = 31, dense), the paired BAM drawn from both."""
    mp = pytest.MonkeyPatch()
    tmp = tmp_path_factory.mktemp("two")
    la, ca = synth.allele_family_library(n_founders=6, alleles_per_founder=10, length=800, snps_mean=8, seed=71)
    lt, ct_ = synth.random_transcript_library(n_seqs=300, mean_len=1500, family_frac=0.4, seed=72)
    ja, jt = _dump(la, tmp / "alle.json"), _dump(lt, tmp / "tx.json")
    it = _index(jt, tmp / "tx.nb200idx", 31, mp, "0.9")
    ia = _index(ja, tmp / "alle.nb200idx", 20, mp)
    bam = _pairs_bam(tmp, ca[:30] + ct_[:30], 30_000, 73)
    mp.undo()
    return tmp, ja, jt, ia, it, bam


def test_files_counts_paired_two_libraries_trim(engine, two_libs, monkeypatch, tmp_path):
    """align --counts --output on paired input, two libraries and --trim: a JSON and an index library in one call (k = 20 and
    31) give the per-read and counts TSVs of the two JSON libraries; so do *_multi calls on {0, 0} (and {0, 1})."""
    import torch
    _, ja, jt, ia, it, bam = two_libs
    want = [_json_lib(engine, ja, 20, None, monkeypatch), _json_lib(engine, jt, 31, "0.9", monkeypatch)]
    got = [engine.load_library(ja), engine.load_library(it)]
    for lg, t in zip(want + got, [(70, 0.6), (90, 0.4)] * 2):
        lg.set_trim(*t)
    res = {}
    for tag, libs in (("json", want), ("index", got)):
        outs = [str(tmp_path / ("%s.%d.tsv" % (tag, i))) for i in range(2)]
        cnts = [str(tmp_path / ("%s.%d.counts.tsv" % (tag, i))) for i in range(2)]
        o3 = engine.align_files_counts([bam], libs, cnts, outs)
        res[tag] = (o3, [_read(p) for p in outs + cnts])
    assert res["json"] == res["index"] and min(x[0] for x in res["json"][0]) > 5000
    # the frontend and the multi-context entries: k unset -> 20 for the JSON, 31 from the index file
    ref = "%s,%s" % (ja, it)
    devsets = [None, [0, 0]] + ([[0, 1]] if torch.cuda.device_count() >= 2 else [])
    for devs in devsets:
        out, cnt = str(tmp_path / "f.tsv"), str(tmp_path / "f_counts.tsv")
        assert frontend.align(ref, out, [bam], 4, "unstranded", "70:0.6,90:0.4", None, engine=None if devs else engine, gpus=devs,
                              counts=cnt) == 0
        libs = ref.split(",")
        data = [_read(p) for p in frontend._per_library_paths(out, libs) + frontend._per_library_paths(cnt, libs)]
        assert data == res["json"][1], devs


def test_fastq_to_counts_and_aligner_from_index(engine, two_libs, tmp_path):
    tmp, ja, jt, ia, it, _ = two_libs
    codes = synth.allele_family_library(n_founders=6, alleles_per_founder=10, length=800, snps_mean=8, seed=71)[1]
    f1, f2, wlp, _, _, _ = _tenx(tmp_path, codes, 40_000, 74, clustered=0.3)
    outs = {}
    for tag, ref, devs in (("json", ja, None), ("index", ia, None), ("index_multi", ia, [0, 0])):
        cnt = str(tmp_path / ("%s.counts.tsv" % tag))
        assert frontend.fastq_to_counts(ref, f1, f2, wlp, cnt, 4, engine=None if devs else engine, gpus=devs) == 0
        outs[tag] = _read(cnt)
    assert len(outs["json"]) > 1000 and outs["json"] == outs["index"] == outs["index_multi"]
    # the drop-in aligner: -r LIB.nb200idx (no -k: the index's own) equals -r LIB.json at the same k
    bam = two_libs[5]
    a, b = str(tmp_path / "a.tsv"), str(tmp_path / "b.tsv")
    for r, o, extra in ((jt, a, ["-k", "31"]), (it, b, [])):
        p = subprocess.run([ALIGNER, "--input", bam, "-c", "4", "--strand_filter", "unstranded", "-r", r, "-o", o] + extra,
                           capture_output=True, text=True, env=dict(os.environ, NB200_TABLE_LF="0.9"))
        assert p.returncode == 0, p.stderr
    assert _read(a) == _read(b) and len(_read(a)) > 100_000
    p = subprocess.run([ALIGNER, "--input", bam, "-c", "4", "--strand_filter", "unstranded", "-r", it, "-o", a, "-k", "20"],
                       capture_output=True, text=True)
    assert p.returncode == 1 and "k = 31" in p.stderr and "k = 20" in p.stderr


def test_k_mismatch_and_damaged_image(engine, two_libs, tmp_path):
    tmp, ja, jt, ia, it, bam = two_libs
    with pytest.raises(NimbleB200Error) as e:
        engine.load_library(it, k=20)
    assert e.value.code == EINVAL and "k = 31" in str(e.value) and "k = 20" in str(e.value)
    assert engine.load_library(it, k=31).info["n_refs"] == 300
    # one byte flipped inside the device image (header and host sections intact): refused by the device checksum
    data = bytearray(_read(ia))
    img_off = int.from_bytes(data[296 + 72:296 + 80], "little")
    data[img_off + len(data[img_off:]) // 2] ^= 0x04
    bad = str(tmp_path / "bad.nb200idx")
    with open(bad, "wb") as f:
        f.write(bytes(data))
    r1, truth = synth.sample_reads(synth.allele_family_library(n_founders=6, alleles_per_founder=10, length=800, snps_mean=8,
                                                               seed=71)[1], 20_000, read_len=90, seed=75)
    before = engine.load_library(ja)
    with pytest.raises(NimbleB200Error) as e:
        engine.load_library(bad)
    assert e.value.code == EINVAL and "damaged" in str(e.value) and "checksum" in str(e.value)
    after = engine.load_library(ja)                              # the same context loads the JSON and aligns as before
    assert after.id == before.id + 1
    assert engine.align(after, r1, per_read=True)[1].tobytes() == engine.align(before, r1, per_read=True)[1].tobytes()
    # the multi-context entry reports the damage and writes nothing
    out = str(tmp_path / "m.tsv")
    assert frontend.align(bad, out, [bam], 4, "unstranded", "", None, gpus=[0, 0]) == 1
    assert not os.path.exists(out)
