"""Native `report -s` (nb200_summarize_file, Engine.summarize_file) against the Python path, frontend.summarize_fields_tsv:
the pandas-generated golden cases, a seeded differential over generated per-read TSVs, scale cases, the CLI end to end
and the C ABI's errors (DESIGN.md §2.13)."""
import ctypes as ct
import gzip
import json
import os
import random

import numpy as np
import pytest

from nimble_b200 import _lib, frontend

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
NA_TOKENS = sorted(frontend._PANDAS_NA)
BASE = ["nimble_features", "nimble_score", "r1_QNAME", "r1_CB", "r1_UB", "r1_GN", "r1_POS"]


def _native(engine, path, cols, out):
    return engine.summarize_file(str(path), cols, str(out))


def _python(path, cols, out):
    frontend.summarize_fields_tsv(str(path), cols, str(out))


def _same(engine, tmp_path, path, cols):
    """Both paths on one file: the same output bytes, or the same KeyError."""
    a, b = tmp_path / "native.tsv", tmp_path / "python.tsv"
    try:
        _python(path, cols, b)
    except KeyError as e:
        with pytest.raises(KeyError) as got:
            _native(engine, path, cols, a)
        assert got.value.args == e.args
        return None
    rows, umis = _native(engine, path, cols, a)
    assert a.read_bytes() == b.read_bytes(), (path, cols)
    return rows, umis


# ---- the 60 golden cases ------------------------------------------------------------------------------
def test_golden_cases_byte_identical(engine, tmp_path):
    with open(os.path.join(HERE, "golden", "summarize_cases.json")) as f:
        d = json.load(f)
    n = 0
    for c in d["cases"]:
        inp, out = tmp_path / ("%s.tsv" % c["id"]), tmp_path / "o.tsv"
        with open(inp, "w") as f:
            f.write("\t".join(d["header"]) + "\n")
            for r in c["rows"]:
                f.write("\t".join(r) + "\n")
        if c["expected"] is None:
            with pytest.raises(KeyError):
                _native(engine, inp, c["columns"], out)
            _same(engine, tmp_path, inp, c["columns"])
            continue
        _native(engine, inp, c["columns"], out)
        assert out.read_text() == c["expected"]["text"], c["id"]
        n += 1
    assert n >= 50


# ---- seeded differential ------------------------------------------------------------------------------
def _int_cell(rng):
    k = rng.randrange(8)
    if k == 0:
        return str(rng.randrange(-5, 6))
    if k == 1:
        return rng.choice(["+", "-", ""]) + "0" * rng.randrange(1, 3) + str(rng.randrange(0, 20))
    if k == 2:
        return rng.choice(["-0", "+0", "000", "-000"])
    if k == 3:
        return str(rng.choice([-1, 1]) * rng.randrange(2 ** 64, 2 ** 70))        # beyond 64 bits
    if k == 4:
        return str(rng.randrange(10 ** 17, 10 ** 19))                           # on both sides of 18 digits
    return str(rng.randrange(0, 12))


def _float_cell(rng):
    k = rng.randrange(10)
    if k == 0:
        return rng.choice(["1e5", "1E+05", "2.5e-7", "1e16", "1e-5", "1e22", ".5", "5.", "-.25e1", "1e400", "-1e-400"])
    if k == 1:
        return rng.choice(["inf", "-inf", "Infinity", "+INF", "-iNfInItY"])
    if k == 2:
        return rng.choice(["-0.0", "0.0", "-0", "0e0", "+0.000"])
    if k == 3:
        return rng.choice([" 2", "3 ", "\x0b4", "5\x0c", " 1.5 "])                 # padded: never an int column
    if k == 4:
        return repr(rng.uniform(-1e6, 1e6))
    if k == 5:
        return rng.choice(["NAN", "+nan", "Nan", "-NAN"])                          # NaN texts that are not NA tokens
    return "%d.%d" % (rng.randrange(0, 4), rng.randrange(0, 3))


def _string_cell(rng):
    k = rng.randrange(8)
    if k == 0:
        return rng.choice(["1_000", "_5", "1__2", "1.5_0"])                        # '_' never parses
    if k == 1:
        return rng.choice(['a"b', '"q"', '""'])
    if k == 2:
        return rng.choice(["HLA-A", "HLA-B", "HLA-A,HLA-B", "é", "zz", "Z", "a b"])
    if k == 3:
        return rng.choice(["0x10", "1e", "e5", "--1", "+-1", "1.2.3", "inf5", "nan1"])
    return rng.choice(["g1", "g2", "g3", "g10", "x"])


def _umi_cell(rng, kind):
    if kind == "int":
        return str(rng.randrange(0, 30)) if rng.random() < 0.9 else rng.choice(["007", "+7", "-3", "-0"])
    if kind == "float":
        return rng.choice(["1.5", "2", "-0.0", "0", "1e3", "inf", "-inf", "0.1", "1000"])
    if kind == "long":
        return str(rng.choice([2 ** 65, -(2 ** 66), 3, 10 ** 20, -5]))
    return rng.choice(["AACC", "AAGT", "TTTT", "ACGTACGTACGT", "GG", "N", "A"]) + rng.choice(["", "", "-1"])


def make_case(seed):
    """One generated per-read TSV: (file bytes, -s columns, gzip or not)."""
    rng = random.Random(seed)
    header = list(BASE) + ["X", "Y"]
    if rng.random() < 0.15:
        header.append(rng.choice(["X", "r1_GN", "umi"]))                           # duplicate names: the last one wins
    rng.shuffle(header)
    umi_kind = rng.choice(["str", "str", "int", "float", "long", "none"])
    col_kind = {h: rng.choice(["int", "int_blank", "float", "string", "mixed", "na"]) for h in header}
    n_rows = rng.choice([0, 1, 3, 20, 60, 200])
    na_rate = rng.choice([0.0, 0.05, 0.3])
    tie_umis = rng.random() < 0.3
    lines = []
    for i in range(n_rows):
        row = []
        for h in header:
            if h in ("r1_UB", "umi"):
                if umi_kind == "none" or rng.random() < na_rate:
                    v = rng.choice(NA_TOKENS)
                else:
                    v = _umi_cell(rng, umi_kind)
                if tie_umis:
                    v = _umi_cell(random.Random(i // 4), umi_kind) if umi_kind != "none" else v
            else:
                k = col_kind[h]
                if k == "na" or (k != "int" and rng.random() < na_rate) or (k == "int_blank" and rng.random() < 0.1):
                    v = rng.choice(NA_TOKENS)
                elif k in ("int", "int_blank"):
                    v = _int_cell(rng)
                elif k == "float":
                    v = rng.choice([_float_cell, _int_cell])(rng)
                elif k == "string":
                    v = _string_cell(rng)
                else:
                    v = rng.choice([_int_cell, _float_cell, _string_cell])(rng)
                if tie_umis and h == "Y":
                    v = "ab"[i % 2]                                                 # equal counts inside a UMI
            row.append(v)
        if rng.random() < 0.05:
            row = row[:rng.randrange(0, len(row))]                                  # short row: empty cells
        elif rng.random() < 0.05:
            row = row + ["extra", "cells"]
        lines.append("\t".join(row) if row or rng.random() < 0.5 else "")
    eol = rng.choice(["\n", "\n", "\r\n", "\r", "mixed"])

    def end():
        return rng.choice(["\n", "\r\n", "\r"]) if eol == "mixed" else eol
    text = "\t".join(header) + end() + "".join(x + end() for x in lines)
    if lines and rng.random() < 0.2:
        text = text[:-2] if text.endswith("\r\n") else text[:-1]                        # no line end after the last row
    pool = [h for h in header if h not in ("r1_UB", "umi")] + ["r1_UB"]
    cols = rng.sample(pool, rng.randrange(1, 4))
    if rng.random() < 0.2:
        cols.append(cols[0])                                                        # the same column twice
    if rng.random() < 0.1:
        cols.append(rng.choice(["features", "cb", "umi"]))                          # names after renaming
    if rng.random() < 0.03:
        cols.append("missing_column")
    return text.encode(), cols, rng.random() < 0.15


def _write_case(tmp_path, i, data, gz):
    p = tmp_path / ("case%d.tsv%s" % (i, ".gz" if gz else ""))
    if gz:
        with gzip.open(p, "wb") as f:
            f.write(data)
    else:
        p.write_bytes(data)
    return p


def test_differential_against_python(engine, tmp_path):
    n = int(os.environ.get("NB200_FUZZ_CASES", "300"))
    checked = 0
    for i in range(n):
        data, cols, gz = make_case(1000 + i)
        p = _write_case(tmp_path, i, data, gz)
        r = _same(engine, tmp_path, p, cols)
        if r is not None:
            checked += 1
        p.unlink()
    assert checked >= 200


def test_nan_texts_in_value_columns(engine, tmp_path):
    """A NaN that is not an NA token is one value per text, as Python's float objects are (DESIGN.md §2.13)."""
    p = tmp_path / "nan.tsv"
    p.write_text("r1_UB\tX\nu\tNAN\nu\tNAN\nu\t+nan\nu\t1\nv\tNaN\n")
    _same(engine, tmp_path, p, ["X"])
    assert (tmp_path / "native.tsv").read_text() == "umi\tX\nu\tnan(2); nan(1); 1.0(1)\nv\t\n"


def test_reading_rules(engine, tmp_path):
    """Lone CR and CRLF end lines, short rows pad, an empty line is a row of NA cells (so the int columns become float
    columns), equal values merge, quoted output cells."""
    p = tmp_path / "r.tsv"
    p.write_bytes(b"r1_UB\tX\tY\n9\t005\ta\"b\r10\t+5\r\n9\t5\n\n9\n10\t-0\t\"\n")
    rows, umis = _same(engine, tmp_path, p, ["X", "Y"])
    assert (rows, umis) == (6, 2)
    assert (tmp_path / "native.tsv").read_text() == 'umi\tX\tY\n9.0\t5.0(2)\t"a""b(1)"\n10.0\t5.0(1); 0.0(1)\t"""(1)"\n'


def _big_tsv(path, n, rng, umi=None, qname=False):
    """A per-read TSV shaped like align's: n rows, seeded."""
    cells = np.array(["".join(rng.choice(list("ACGT"), 16)) + "-1" for _ in range(500)])
    umis = np.array(["".join(x) for x in rng.choice(list("ACGT"), (4096, 10))])
    feats = np.array(["A", "B", "A,B", "C", "D"])
    gn = np.array(["HLA-A", "HLA-B", "", "CD3E"])
    u = np.full(n, umi) if umi is not None else umis[rng.integers(0, len(umis), n)]
    cols = [feats[rng.integers(0, 5, n)], np.full(n, "1"), np.char.add("read", np.arange(n).astype(str)),
            cells[rng.integers(0, 500, n)], u, gn[rng.integers(0, 4, n)], rng.integers(1, 10 ** 6, n).astype(str)]
    with open(path, "w") as f:
        f.write("\t".join(BASE) + "\n")
        f.write("\n".join("\t".join(r) for r in zip(*cols)))
        f.write("\n")


@pytest.mark.parametrize("shape", ["2M_rows", "one_umi_1M_rows", "one_umi_many_values", "all_distinct_qname"])
def test_scale_against_python(engine, tmp_path, shape):
    rng = np.random.default_rng(7)
    p = tmp_path / "big.tsv"
    if shape == "2M_rows":
        _big_tsv(p, 2_000_000, rng)
        cols = ["r1_GN", "r1_POS", "nimble_features"]
    elif shape == "one_umi_1M_rows":
        _big_tsv(p, 1_000_000, rng, umi="ACGTACGTAC")
        cols = ["r1_GN", "nimble_features"]
    elif shape == "one_umi_many_values":                          # > 65 536 distinct values inside one UMI
        _big_tsv(p, 300_000, rng, umi="ACGTACGTAC")
        cols = ["r1_POS"]
    else:
        _big_tsv(p, 500_000, rng)
        cols = ["r1_QNAME", "r1_CB"]
    rows, umis = _same(engine, tmp_path, p, cols)
    assert rows > 0 and umis > 0


def test_cli_end_to_end(tmp_path):
    """align --output on a seeded BAM, then `report -s` through the CLI: native and Python summaries are identical."""
    import subprocess
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(HERE), "scripts"))
    import file_bench
    from nimble_b200 import synth
    lib, codes = synth.allele_family_library(n_founders=8, alleles_per_founder=20, length=700, snps_mean=10, seed=11)
    r1, truth = synth.sample_reads(codes, 20000, read_len=90, seed=12)
    key = synth.barcodes_10x(20000, n_cells=200, seed=12, truth=truth)
    with open(tmp_path / "lib.json", "w") as f:
        json.dump(lib, f)
    file_bench.write_bam(str(tmp_path / "in.bam"), r1, key)
    env = dict(os.environ, PYTHONPATH=os.path.dirname(HERE))
    cli = [sys.executable, "-m", "nimble_b200"]
    cols = ["r1_GN", "nimble_features", "r1_CB", "nimble_score"]
    subprocess.run(cli + ["align", "--reference", "lib.json", "--output", "per_read.tsv", "--input", "in.bam"], cwd=tmp_path, env=env,
                   check=True)
    subprocess.run(cli + ["report", "-i", "per_read.tsv", "-o", "counts.tsv", "-s", ",".join(cols)], cwd=tmp_path, env=env, check=True)
    _python(tmp_path / "per_read.tsv", cols, tmp_path / "py.tsv")
    got = (tmp_path / "summarize.counts.tsv").read_bytes()
    assert got == (tmp_path / "py.tsv").read_bytes() and got.count(b"\n") > 10


# ---- C ABI --------------------------------------------------------------------------------------------
def test_abi_errors_and_out2(engine, tmp_path):
    L = engine.L
    p = tmp_path / "a.tsv"
    p.write_text("r1_UB\tX\nu\t1\nv\t2\nNA\t3\n")
    cols = (ct.c_char_p * 1)(b"X")
    out2 = (ct.c_uint64 * 2)()
    assert L.nb200_summarize_file(engine.ctx, str(p).encode(), cols, 1, str(tmp_path / "o.tsv").encode(), out2) == _lib.OK
    assert list(out2) == [3, 2]
    assert L.nb200_summarize_file(engine.ctx, str(p).encode(), cols, 1, str(tmp_path / "o.tsv").encode(), None) == _lib.OK
    assert L.nb200_summarize_file(engine.ctx, str(tmp_path / "nope.tsv").encode(), cols, 1, b"o", out2) == _lib.EIO
    bad = (ct.c_char_p * 1)(b"r1_CB")
    assert L.nb200_summarize_file(engine.ctx, str(p).encode(), bad, 1, b"o", out2) == _lib.EINVAL
    assert b"missing column: cb" in L.nb200_last_error(engine.ctx)
    assert L.nb200_summarize_file(engine.ctx, None, cols, 1, b"o", out2) == _lib.EINVAL
    assert L.nb200_summarize_file(engine.ctx, str(p).encode(), None, 1, b"o", out2) == _lib.EINVAL
    assert L.nb200_summarize_file(engine.ctx, str(p).encode(), cols, 1, None, out2) == _lib.EINVAL
    assert L.nb200_summarize_file(None, str(p).encode(), cols, 1, b"o", out2) == _lib.EINVAL
    with pytest.raises(KeyError) as e:
        engine.summarize_file(p, ["nimble_features"], tmp_path / "o.tsv")
    assert e.value.args == ("features",)
    q = tmp_path / "noumi.tsv"
    q.write_text("r1_UB\tX\nNA\t1\n\t2\n")
    assert _same(engine, tmp_path, q, ["X"]) == (2, 0)
