"""Host-side mirror of nimble's operator interface (nimble_b200/frontend.py, __main__.py)."""
import gzip
import json
import os
import struct

import numpy as np
import pytest

from nimble_b200 import frontend, synth

HERE = os.path.dirname(os.path.abspath(__file__))
with open(os.path.join(HERE, "golden", "format_goldens.json")) as f:
    FMT = json.load(f)


def test_append_path_string_and_library_name_match_reference():
    for p, a, want in FMT["append_path_string"]:
        assert frontend.append_path_string(p, a) == want
    for n, want in FMT["library_name"]:
        assert frontend.get_library_name_from_filename(n) == want


def test_default_config_json_is_byte_identical_to_reference_dump():
    empty = {"headers": ["reference_genome", "sequence_name", "nt_length", "sequence"], "columns": [[], [], [], []]}
    assert json.dumps([frontend._default_config(), empty], indent=2) == FMT["library_json_empty"]


def test_generate_fasta_and_csv(tmp_path):
    fa = tmp_path / "my_mhc_lib.fasta"
    fa.write_text(">A*01 some description\nACGTAC\nGTAC\n>B*02\nTTTT\n\n>\nGG\n")
    out = tmp_path / "lib.json"
    frontend.generate(str(fa), None, str(out))
    text = out.read_text()
    cfg, data = json.loads(text)
    assert text == json.dumps([cfg, data], indent=2)
    assert list(cfg) == list(json.loads(FMT["library_json_empty"])[0])
    assert data["headers"] == ["reference_genome", "sequence_name", "nt_length", "sequence"]
    assert data["columns"] == [["my mhc lib"] * 3, ["A*01", "B*02", ""], ["10", "4", "2"], ["ACGTACGTAC", "TTTT", "GG"]]
    # CSV with sequences + metadata column
    cs = tmp_path / "meta_lib.csv"
    cs.write_text('name,gene,sequence\nA*01,A,ACGTACGTAC\n"B*02",B,TTTT\n')
    frontend.generate(str(cs), None, str(out))
    cfg, data = json.loads(out.read_text())
    assert data["headers"] == ["reference_genome", "sequence_name", "nt_length", "sequence", "gene"]
    assert data["columns"][1] == ["A*01", "B*02"] and data["columns"][4] == ["A", "B"] and data["columns"][2] == ["10", "4"]
    # CSV metadata + FASTA sequences (collate): CSV rows win, sequences copied by name
    cs2 = tmp_path / "meta_only.csv"
    cs2.write_text("name,gene\nB*02,B\nA*01,A\n,N\n")
    frontend.generate(str(fa), str(cs2), str(out))
    cfg, data = json.loads(out.read_text())
    assert data["columns"][1] == ["B*02", "A*01", ""] and data["columns"][3] == ["TTTT", "ACGTACGTAC", "GG"]
    with pytest.raises(ValueError):
        frontend.generate(str(tmp_path / "x.fa"), None, str(out))


def write_bam(path, records):
    """records: (name, flag, seq, {tag: str}[, phred qualities]) -> minimal unaligned BAM (one gzip member)."""
    body = b"BAM\x01" + struct.pack("<i", 0) + struct.pack("<i", 0)
    code = {c: i for i, c in enumerate("=ACMGRSVTWYHKDBN")}
    for rec_in in records:
        name, flag, seq, tags = rec_in[:4]
        qual = bytes(int(x) for x in rec_in[4]) if len(rec_in) > 4 else b"\xff" * len(seq)
        nm = name.encode() + b"\x00"
        packed = bytearray((len(seq) + 1) // 2)
        for i, ch in enumerate(seq):
            packed[i // 2] |= code[ch] << (4 if i % 2 == 0 else 0)
        tagb = b"".join(t.encode() + b"Z" + v.encode() + b"\x00" for t, v in tags.items())
        core = struct.pack("<iiBBHHHiiii", -1, -1, len(nm), 0, 4680, 0, flag, len(seq), -1, -1, 0)
        rec = core + nm + bytes(packed) + qual + tagb
        body += struct.pack("<i", len(rec)) + rec
    with gzip.open(path, "wb") as g:
        g.write(body)


def test_bam_and_fastq_readers(tmp_path):
    bam = tmp_path / "x.bam"
    write_bam(str(bam), [("q1", 77, "ACGTN", {"CB": "AAAC", "UB": "GG", "GN": "geneX"}), ("q1", 141, "TTGCA", {"CB": "AAAC", "UB": "GG"}),
                         ("q2", 77, "ACG", {}), ("q2", 141, "CCC", {})])
    d = frontend.load_reads([str(bam)])
    assert d["names"] == ["q1", "q2"] and d["r1"] == ["ACGTN", "ACG"] and d["r2"] == ["TTGCA", "CCC"]
    assert d["cb"] == ["AAAC", ""] and d["ub"] == ["GG", ""]
    fq = tmp_path / "r1.fastq.gz"
    with gzip.open(fq, "wt") as g:
        g.write("@r1 desc\nACGT\n+\nIIII\n@r2\nGGA\n+\nIII\n")
    d = frontend.load_reads([str(fq)])
    assert d["names"] == ["r1", "r2"] and d["r1"] == ["ACGT", "GGA"] and d["r2"] is None and d["cb"] is None


def test_cli_parses_the_reference_flags(tmp_path, capsys):
    from nimble_b200.__main__ import main
    main(["download"])
    assert "nothing to download" in capsys.readouterr().out
    fa = tmp_path / "l.fasta"
    fa.write_text(">a\nACGT\n")
    main(["generate", "--file", str(fa), "--output_path", str(tmp_path / "l.json")])
    assert json.loads((tmp_path / "l.json").read_text())[1]["columns"][1] == ["a"]


@pytest.mark.gpu
def test_report_reproduces_pandas_reference_tsv(engine, tmp_path, capsys):
    gold = json.load(open(os.path.join(HERE, "golden", "a6_pandas_cases.json")))
    n = 0
    for c in gold["cases"]:
        if c["reference_error"]:
            continue
        inp, out = tmp_path / "in.tsv", tmp_path / "out.tsv"
        with open(inp, "w") as f:
            f.write("nimble_features\tnimble_score\tr1_CB\tr1_UB\n")
            for feats, score, cb, umi in c["rows"]:
                f.write("%s\t%s\t%s\t%s\n" % (feats, repr(score) if isinstance(score, float) else score, cb, umi))
        for native in (True, False):          # native parser/writer (nb200_report_file) and the Python mirror
            frontend.report(str(inp), str(out), None, c["threshold"], c["disable_thresholding"], engine=engine, native=native)
            assert out.read_text() == (c["expected_tsv"] or ""), (c["id"], native)
            log = capsys.readouterr().out
            if "Dropped" in c["reference_stdout"]:
                assert c["reference_stdout"].strip() in log
        n += 1
    assert n > 250


@pytest.mark.gpu
def test_align_then_report_end_to_end(engine, tmp_path):
    from oracle import oracle as O
    from helpers import oracle_counts, to_concat
    lib, codes = synth.allele_family_library(n_founders=4, alleles_per_founder=6, length=400, snps_mean=6, seed=131)
    fa = tmp_path / "mhc_lib.fasta"
    names, seqs = lib[1]["columns"][1], lib[1]["columns"][3]
    fa.write_text("".join(">%s\n%s\n" % (n, s) for n, s in zip(names, seqs)))
    libjson = tmp_path / "mhc_lib.json"
    frontend.generate(str(fa), None, str(libjson))
    r1, truth = synth.sample_reads(codes, 3000, read_len=90, seed=132)
    key = synth.barcodes_10x(len(r1), n_cells=12, seed=133, truth=truth)
    reads = ["".join(map(chr, r)) for r in r1]
    cbs = [synth.unpack_barcode(int(k) >> 32, 16) for k in key]
    ubs = [synth.unpack_barcode(int(k) & 0xFFFFFF, 12) for k in key]
    bam = tmp_path / "in.bam"
    write_bam(str(bam), [("read%d" % i, 4, reads[i], {"CB": cbs[i], "UB": ubs[i]}) for i in range(len(reads))])
    out = tmp_path / "out.tsv.gz"
    rc = frontend.align(str(libjson), str(out), [str(bam)], 2, "unstranded", "", None, engine=engine)
    assert rc == 0
    counts = tmp_path / "counts.tsv"
    frontend.report(str(out), str(counts), None, 0.05, False, engine=engine)
    # oracle: same library / reads / keys
    lo = O.Library(json.loads(libjson.read_text()))
    ro, fo = O.align(lo, to_concat(r1))
    cell, cnt, off, ids, dropped = oracle_counts(lo, ro, fo, key)
    want = "".join("%s\t%d\t%s\n" % (",".join(lo.features[j] for j in ids[off[i]:off[i + 1]]), cnt[i], synth.unpack_barcode(int(cell[i]), 16))
                   for i in range(len(cell)))
    assert counts.read_text() == want and len(cell) > 20
    # FASTQ (bulk) input, two libraries -> two outputs named like the reference does
    fq = tmp_path / "r.fastq"
    fq.write_text("".join("@r%d\n%s\n+\n%s\n" % (i, reads[i], "I" * 90) for i in range(500)))
    lib2 = tmp_path / "second.json"
    lib2.write_text(libjson.read_text())
    rc = frontend.align("%s,%s" % (libjson, lib2), str(tmp_path / "bulk.tsv"), [str(fq)], 1, "unstranded", "", None, engine=engine)
    assert rc == 0 and (tmp_path / "bulk.mhc_lib.tsv").exists() and (tmp_path / "bulk.second.tsv").exists()
    lines = (tmp_path / "bulk.mhc_lib.tsv").read_text().splitlines()
    assert lines[0] == "nimble_features\tnimble_score" and sum(int(l.split("\t")[1]) for l in lines[1:]) == int((ro["n_feat"][:500] > 0).sum())
    # failure -> non-zero return code, inputs untouched
    assert frontend.align(str(tmp_path / "missing.json"), str(tmp_path / "o.tsv"), [str(fq)], 1, "unstranded", "", None, engine=engine) != 0
    assert frontend.align(str(libjson), str(tmp_path / "o.tsv"), [str(fq)], 1, "sideways", "", None, engine=engine) != 0


@pytest.mark.gpu
def test_aligner_executable_with_the_reference_argv(engine, tmp_path):
    """The `aligner` binary is invoked exactly as nimble/__main__.py:177-196 does: its TSVs must equal
    the Python front end's (same engine underneath) and feed `report` to the oracle's counts."""
    import gzip as gz
    import subprocess
    from oracle import oracle as O
    from helpers import oracle_counts, to_concat
    exe = os.path.join(os.path.dirname(HERE), "nimble_b200", "aligner")
    assert os.path.exists(exe), "nimble_b200/aligner not built"
    lib, codes = synth.allele_family_library(n_founders=4, alleles_per_founder=6, length=400, snps_mean=6, seed=171)
    lib_b, _ = synth.allele_family_library(n_founders=2, alleles_per_founder=5, length=300, seed=172, name_prefix="KIR")
    p_a, p_b = tmp_path / "mhc_lib.json", tmp_path / "kir.json"
    p_a.write_text(json.dumps(lib, indent=2)); p_b.write_text(json.dumps(lib_b, indent=2))
    r1, r2, truth = synth.sample_pairs(codes, 1500, read_len=100, insert_mean=220, seed=173)
    key = synth.barcodes_10x(len(r1), n_cells=9, seed=174, truth=truth)
    s1 = ["".join(map(chr, r)) for r in r1]; s2 = ["".join(map(chr, r)) for r in r2]
    cbs = [synth.unpack_barcode(int(k) >> 32, 16) for k in key]
    ubs = [synth.unpack_barcode(int(k) & 0xFFFFFF, 12) for k in key]
    recs = []
    for i in range(len(s1)):
        tags = {"CB": cbs[i], "UB": ubs[i], "UR": ubs[i]} if i % 50 else {}
        recs.append(("q%d" % i, 77, s1[i], tags)); recs.append(("q%d" % i, 141, s2[i], tags))
    bam = tmp_path / "in.bam"
    write_bam(str(bam), recs)
    # argv exactly as the reference builds it for two libraries (out.tsv.gz -> out.<stem>.tsv.gz)
    o_a, o_b = tmp_path / "out.mhc_lib.tsv.gz", tmp_path / "out.kir.tsv.gz"
    argv = [exe, "--input", str(bam), "-c", "4", "--strand_filter", "unstranded", "-r", str(p_a), "-o", str(o_a),
            "-r", str(p_b), "-o", str(o_b)]
    out = subprocess.run(argv, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    rc = frontend.align("%s,%s" % (p_a, p_b), str(tmp_path / "py.tsv.gz"), [str(bam)], 4, "unstranded", "", None, engine=engine,
                        native=False)       # file parsing + TSV writing in Python: cross-checks the native file code
    assert rc == 0
    rc = frontend.align("%s,%s" % (p_a, p_b), str(tmp_path / "nat.tsv.gz"), [str(bam)], 4, "unstranded", "", None, engine=engine)
    assert rc == 0 and gz.open(tmp_path / "nat.mhc_lib.tsv.gz", "rt").read() == gz.open(o_a, "rt").read()
    assert gz.open(o_a, "rt").read() == gz.open(tmp_path / "py.mhc_lib.tsv.gz", "rt").read()
    assert gz.open(o_b, "rt").read() == gz.open(tmp_path / "py.kir.tsv.gz", "rt").read()
    counts = tmp_path / "counts.tsv"
    frontend.report(str(o_a), str(counts), None, 0.05, False, engine=engine)
    lo = O.Library(lib)
    ro, fo = O.align(lo, to_concat(r1), to_concat(r2))
    keyed = key.copy(); keyed[::50] = np.uint64(0xFFFFFFFFFFFFFFFF)
    cell, cnt, off, ids, dropped = oracle_counts(lo, ro, fo, keyed)
    want = "".join("%s\t%d\t%s\n" % (",".join(lo.features[j] for j in ids[off[i]:off[i + 1]]), cnt[i], synth.unpack_barcode(int(cell[i]), 16))
                   for i in range(len(cell)))
    assert counts.read_text() == want
    # FASTQ(.gz) pair -> bulk table; error paths -> non-zero exit code and no output
    f1, f2 = tmp_path / "r1.fastq.gz", tmp_path / "r2.fastq"
    with gz.open(f1, "wt") as g:
        g.write("".join("@r%d x\n%s\n+\n%s\n" % (i, s1[i], "I" * 100) for i in range(400)))
    f2.write_text("".join("@r%d\n%s\n+\n%s\n" % (i, s2[i], "I" * 100) for i in range(400)))
    o_c = tmp_path / "bulk.tsv"
    out = subprocess.run([exe, "--input", str(f1), "--input", str(f2), "-c", "2", "--strand_filter", "unstranded", "-r", str(p_a), "-o", str(o_c)],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    lines = o_c.read_text().splitlines()
    assert lines[0] == "nimble_features\tnimble_score" and sum(int(l.split("\t")[1]) for l in lines[1:]) == int((ro["n_feat"][:400] > 0).sum())
    bad = subprocess.run([exe, "--input", str(bam), "-c", "1", "--strand_filter", "sideways", "-r", str(p_a), "-o", str(tmp_path / "no.tsv")],
                         capture_output=True, text=True, timeout=120)
    assert bad.returncode != 0 and not (tmp_path / "no.tsv").exists()
    bad = subprocess.run([exe, "--input", str(tmp_path / "missing.bam"), "-c", "1", "--strand_filter", "unstranded", "-r", str(p_a), "-o", str(tmp_path / "no.tsv")],
                         capture_output=True, text=True, timeout=120)
    assert bad.returncode != 0 and not (tmp_path / "no.tsv").exists()


def _summarize_cases():
    with open(os.path.join(os.path.dirname(__file__), "golden", "summarize_cases.json")) as f:
        return json.load(f)


def test_summarize_matches_pandas_reference(tmp_path):
    """`report -s`: summarize_fields (nimble/__main__.py:295-297) against outputs of the reference's own
    pandas code (tests/golden/make_summarize_golden.py)."""
    d = _summarize_cases()
    n = 0
    for c in d["cases"]:
        if c["expected"] is None:
            continue
        inp, out = str(tmp_path / "in.tsv"), str(tmp_path / "summary.tsv")
        with open(inp, "w") as f:
            f.write("\t".join(d["header"]) + "\n")
            for r in c["rows"]:
                f.write("\t".join(r) + "\n")
        frontend.summarize_fields_tsv(inp, c["columns"], out)
        assert open(out).read() == c["expected"]["text"], c["id"]
        n += 1
    assert n >= 50


@pytest.mark.gpu
def test_report_with_summarize_writes_both_files(engine, tmp_path, monkeypatch):
    d = _summarize_cases()
    c = next(x for x in d["cases"] if x["expected"] is not None and len(x["rows"]) > 10)
    monkeypatch.chdir(tmp_path)                       # the reference writes "summarize." + output (relative)
    with open("in.tsv", "w") as f:
        f.write("\t".join(d["header"]) + "\n")
        for r in c["rows"]:
            f.write("\t".join(r) + "\n")
    frontend.report("in.tsv", "counts.tsv", c["columns"], engine=engine)
    assert os.path.exists("counts.tsv")
    assert open("summarize.counts.tsv").read() == c["expected"]["text"]


def _fnv_reads(d):
    """Same FNV-1a as nb200_host_ingest_stats (csrc/stream.cpp) over the Python reader's view of the file."""
    h = 1469598103934665603
    M = (1 << 64) - 1

    def mix(sv):
        nonlocal h
        for ch in sv.encode("latin-1"):
            h = ((h ^ ch) * 1099511628211) & M
        h = ((h ^ 0xFF) * 1099511628211) & M

    for i in range(len(d["names"])):
        mix(d["names"][i]); mix(d["r1"][i])
        if d["r2"] is not None:
            mix(d["r2"][i])
        if d["cb"] is not None:
            mix(d["cb"][i]); mix(d["ub"][i])
    return h


def _native_ingest(paths, threads=4):
    import ctypes as ct
    from nimble_b200 import _lib
    L = _lib.load()
    arr = (ct.c_char_p * len(paths))(*[p.encode() for p in paths])
    out = (ct.c_uint64 * 6)()
    rc = L.nb200_host_ingest_stats(arr, len(paths), threads, out)
    assert rc == 0, L.nb200_last_error(None)
    return list(out)


def test_native_reader_matches_python_reader(tmp_path):
    """The native FASTQ / BAM reader behind nb200_align_files (block-parallel) sees exactly what the
    plain-Python reader sees: names, mates, CB/UB tags, reverse-strand records restored, secondary skipped."""
    import random
    rng = random.Random(5)
    recs = []
    for i in range(3000):
        name = "read:%d:%s" % (i, "x" * rng.randint(0, 12))
        s1 = "".join(rng.choice("ACGTN") for _ in range(rng.randint(0, 120)))
        s2 = "".join(rng.choice("ACGT") for _ in range(rng.randint(1, 100)))
        tags = {}
        if rng.random() < 0.9:
            tags["CB"] = "".join(rng.choice("ACGT") for _ in range(16))
        if rng.random() < 0.8:
            tags["UB"] = "".join(rng.choice("ACGT") for _ in range(12))
        elif rng.random() < 0.5:
            tags["UR"] = "".join(rng.choice("ACGT") for _ in range(12))
        if rng.random() < 0.3:
            tags["GN"] = "gene%d" % rng.randint(0, 9)
        f1 = 77 if rng.random() < 0.8 else 77 | 0x10
        recs.append((name, f1, s1, tags))
        if rng.random() < 0.05:
            recs.append((name, 0x100 | 77, "ACGT", tags))            # secondary: ignored
        recs.append((name, 141, s2, tags))
    bam = str(tmp_path / "x.bam")
    write_bam(bam, recs)
    d = frontend.load_reads([bam])
    st = _native_ingest([bam])
    assert st[0] == len(d["names"]) == 3000 and st[1] == 1 and st[2] == 1
    assert st[3] == sum(len(x) for x in d["r1"]) and st[4] == sum(len(x) for x in d["r2"])
    assert st[5] == _fnv_reads(d)
    # single-end BAM
    write_bam(bam, [(n, 0, s, t) for (n, f, s, t) in recs if f == 141])
    d = frontend.load_reads([bam])
    st = _native_ingest([bam], threads=1)
    assert st[0] == 3000 and st[1] == 0 and st[5] == _fnv_reads(d)
    # FASTQ pair, one gzipped
    r1, r2 = str(tmp_path / "a.fastq.gz"), str(tmp_path / "b.fastq")
    with gzip.open(r1, "wt") as g:
        for (n, f, s, t) in recs[:500]:
            g.write("@%s extra words\n%s\n+\n%s\n" % (n, s, "I" * len(s)))
    with open(r2, "w") as g:
        for (n, f, s, t) in recs[:500]:
            g.write("@%s/2\n%s\n+\n%s\n" % (n, s[::-1], "I" * len(s)))
    d = frontend.load_reads([r1, r2])
    st = _native_ingest([r1, r2])
    assert st[0] == 500 and st[1] == 1 and st[2] == 0 and st[5] == _fnv_reads(d)


@pytest.mark.gpu
def test_report_file_edge_cases(engine, tmp_path):
    """nb200_report_file: empty / header-only input, pandas' NaN markers, short rows, CRLF, gzip, missing columns."""
    out = tmp_path / "c.tsv"
    empty = tmp_path / "e.tsv"; empty.write_text("")
    assert engine.report_file(str(empty), str(out)) == (0, 0, 0) and out.read_text() == ""
    hdr = "nimble_features\tnimble_score\tr1_CB\tr1_UB\n"
    honly = tmp_path / "h.tsv"; honly.write_text(hdr)
    assert engine.report_file(str(honly), str(out)) == (0, 0, 0) and out.read_text() == ""
    body = ("A,B\t1\tCELL1\tU1\r\n"        # CRLF
            "B\t1\tCELL1\tU1\n"
            "NA\t1\tCELL1\tU2\n"           # features cell is a pandas NaN marker: dropped
            "A\t1\tnull\tU3\n"             # so is this cell barcode
            "A\t\tCELL1\tU4\n"             # missing score
            "A\tx\tCELL1\tU5\n"            # non-numeric score
            "A\t1\n"                        # short row
            "A\t2.5\tCELL2\tU1\n")
    f = tmp_path / "in.tsv.gz"
    with gzip.open(f, "wt", newline="") as g:
        g.write(hdr + body)
    used, n_out, dropped = engine.report_file(str(f), str(out))
    assert used == 3 and dropped == 0
    assert out.read_text() == "B\t1\tCELL1\nA\t1\tCELL2\n"
    for native in (True, False):            # same through the front end, both modes
        frontend.report(str(f), str(out), engine=engine, native=native)
        assert out.read_text() == "B\t1\tCELL1\nA\t1\tCELL2\n"
    bad = tmp_path / "bad.tsv"; bad.write_text("nimble_features\tnimble_score\tr1_CB\nA\t1\tC\n")
    with pytest.raises(Exception):
        engine.report_file(str(bad), str(out))
    with pytest.raises(Exception):
        engine.report_file(str(tmp_path / "missing.tsv"), str(out))


def test_native_reader_pairs_mates_at_any_distance(tmp_path):
    """Coordinate-ordered / shuffled paired BAM: mates are thousands of records apart.  The native reader pairs them
    through a name map like the Python reader (the reference name-sorts first, nimble/__main__.py:345); a record whose
    mate is missing stays a singleton with an empty partner; r1_UB comes from the UB tag only."""
    import random
    rng = random.Random(11)
    recs = []
    for i in range(4000):
        name = "q%d" % i
        tags = {"CB": "".join(rng.choice("ACGT") for _ in range(16))}
        if i % 3:
            tags["UB"] = "".join(rng.choice("ACGT") for _ in range(12))
        else:
            tags["UR"] = "".join(rng.choice("ACGT") for _ in range(12))       # raw UMI only: r1_UB stays empty
        s1 = "".join(rng.choice("ACGT") for _ in range(rng.randint(30, 90)))
        s2 = "".join(rng.choice("ACGT") for _ in range(rng.randint(30, 90)))
        if i % 50 != 7:
            recs.append((name, 77, s1, tags))
        if i % 50 != 9:
            recs.append((name, 141, s2, tags))
    rng.shuffle(recs)
    bam = str(tmp_path / "shuffled.bam")
    write_bam(bam, recs)
    d = frontend.load_reads([bam])
    assert len(d["names"]) == 4000 and sum(1 for u in d["ub"] if u == "") >= 1300
    # the streaming reader emits a pair when its SECOND mate arrives and the singletons at the end of the file (in the
    # order they were read); the Python reader lists pairs by their first mate: same reads, reordered
    seen, done, order = {}, set(), []
    for name, flag, seq, tags in recs:
        if name in seen:
            order.append(name); done.add(name)
        else:
            seen[name] = len(seen)
    order += [n for n in sorted(seen, key=seen.get) if n not in done]
    at = {n: i for i, n in enumerate(d["names"])}
    perm = [at[n] for n in order]
    d2 = {k_: ([v[i] for i in perm] if isinstance(v, list) else v) for k_, v in d.items()}
    for threads in (1, 4):
        st = _native_ingest([bam], threads=threads)
        assert st[0] == 4000 and st[1] == 1
        assert st[3] == sum(len(x) for x in d["r1"]) and st[4] == sum(len(x) for x in d["r2"])
        assert st[5] == _fnv_reads(d2)


def test_native_reader_single_end_bgzf_runs(tmp_path):
    """Single-end BAM in small BGZF blocks (records straddle block boundaries, size fields split across blocks, secondary
    records between the reads): the run-based walk of the streaming reader sees what the Python reader sees."""
    import random
    import zlib
    rng = random.Random(11)
    recs = []
    for i in range(20000):
        s = "".join(rng.choice("ACGTN") for _ in range(rng.randint(1, 150)))
        tags = {"CB": "".join(rng.choice("ACGT") for _ in range(16)), "UB": "".join(rng.choice("ACGT") for _ in range(12))}
        recs.append(("r%d" % i, 16 if rng.random() < 0.3 else 0, s, tags))
        if rng.random() < 0.02:
            recs.append(("r%d" % i, 0x900, "ACGT", tags))                      # secondary + supplementary: skipped
    plain = str(tmp_path / "plain.bam")
    write_bam(plain, recs)
    raw = gzip.open(plain, "rb").read()
    bg = str(tmp_path / "blocks.bam")
    with open(bg, "wb") as f:                                                  # BGZF blocks of odd sizes (a few hundred bytes to 20 kB)
        p = 0
        while p < len(raw):
            n = rng.choice([257, 1021, 4099, 20011])
            blk = raw[p:p + n]
            z = zlib.compressobj(1, zlib.DEFLATED, -15)
            cd = z.compress(blk) + z.flush()
            f.write(bytes([31, 139, 8, 4, 0, 0, 0, 0, 0, 255, 6, 0, 66, 67, 2, 0]) + struct.pack("<H", len(cd) + 25) + cd)
            f.write(struct.pack("<II", zlib.crc32(blk), len(blk)))
            p += n
        f.write(bytes([0x1F, 0x8B, 8, 4, 0, 0, 0, 0, 0, 0xFF, 6, 0, 0x42, 0x43, 2, 0, 0x1B, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0]))
    d = frontend.load_reads([plain])
    want = _fnv_reads(d)
    for path, threads in ((plain, 3), (bg, 1), (bg, 5)):
        st = _native_ingest([path], threads=threads)
        assert st[0] == 20000 and st[1] == 0 and st[2] == 1 and st[3] == sum(len(x) for x in d["r1"])
        assert st[5] == want, path


def test_native_reader_damaged_and_degenerate_files(tmp_path):
    """Header-only, truncated, corrupt, EOF-marker-less, garbage and empty inputs through the streaming reader (dry run):
    an answer or an error code with a message, never a crash; corrupt deflate data is declined by the reader's own decoder
    and diagnosed by zlib."""
    import ctypes as ct
    import sys
    from concurrent.futures import ThreadPoolExecutor
    from nimble_b200 import _lib, synth
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "scripts"))
    import file_bench as fb
    L = _lib.load()

    def ingest(path, threads=3):
        arr = (ct.c_char_p * 1)(str(path).encode())
        out = (ct.c_uint64 * 6)()
        rc = L.nb200_host_ingest_stats(arr, 1, threads, out)
        return rc, list(out), (L.nb200_last_error(None) or b"").decode()

    hdr = tmp_path / "hdr.bam"
    with open(hdr, "wb") as f, ThreadPoolExecutor(2) as ex:
        fb.bgzf_append(f, b"BAM\x01" + struct.pack("<i", 0) + struct.pack("<i", 0), ex)
        f.write(fb.BGZF_EOF)
    rc, st, _ = ingest(hdr)
    assert rc == 0 and st[0] == 0
    lib, codes = synth.allele_family_library(n_founders=2, alleles_per_founder=2, length=300, snps_mean=3.0, seed=1)
    good = tmp_path / "good.bam"
    fb.write_bam_chunked(str(good), codes, 30000, 10, chunk=20000)
    rc, st, _ = ingest(good)
    assert rc == 0 and st[0] == 30000 and st[3] == 30000 * 90
    want = st[5]
    raw = open(good, "rb").read()
    (tmp_path / "noeof.bam").write_bytes(raw[:-28])
    rc, st, _ = ingest(tmp_path / "noeof.bam")
    assert rc == 0 and st[0] == 30000 and st[5] == want
    (tmp_path / "trunc.bam").write_bytes(raw[:len(raw) // 2])
    rc, st, msg = ingest(tmp_path / "trunc.bam")
    assert rc == _lib.EIO and "truncated" in msg
    bad = bytearray(raw)
    for k in range(5):
        bad[len(bad) // 3 + 1000 * k + 57] ^= 0x5A
    (tmp_path / "bad.bam").write_bytes(bytes(bad))
    rc, st, msg = ingest(tmp_path / "bad.bam")
    assert rc == _lib.EIO and "corrupt" in msg
    (tmp_path / "garbage.bam").write_bytes(b"hello world" * 100)
    assert ingest(tmp_path / "garbage.bam")[0] == _lib.EINVAL
    (tmp_path / "empty.bam").write_bytes(b"")
    assert ingest(tmp_path / "empty.bam")[0] == _lib.EINVAL
