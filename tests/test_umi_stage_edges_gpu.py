"""The UMI stage on both sides of each of its size switches, with and without `--correct-umis`.

aggregate() picks its path from the sizes of its input: the per-group insertion sort up to 48 rows a group
(kLocalSortMax), the global token sort above; thread-local working sets up to 8 rows and 16 names (kSmallRows,
kSmallNames); 4, 3, 2 or 1 token columns per radix key by feature count; a stage-2 key of bits_for(D) + bits_for(C) + 1
bits; a correction table sized from the selected rows.  Every case (tests/umi_stage_cases.py, placed on its edge by
tests/test_umi_stage_edges.py) goes through nb200_umi_counts and is compared with the C oracle (oracle.a6_ids) on
cell, count, lists and dropped UMIs; with correction the keys go through oracle/umi_correct_py.py first.  Cases with
string rows also go through the per-read TSV route (nb200_report_file: the native reader and UMI interning) and are
compared byte for byte with the string oracles."""
import json
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "scripts"))

import umi_stage_cases as U
from nimble_b200 import synth
from oracle.a6_py import report_counts
from oracle.umi_correct_py import correct_umis

pytestmark = pytest.mark.gpu

_libs = {}


def lib_for(engine, names):
    k = (id(engine), len(names), hash(tuple(names)))
    if k not in _libs:
        _libs[k] = engine.load_feature_names(names)
    return _libs[k]


def check(engine, case, thr, dis, correct=False):
    t = engine.umi_counts(lib_for(engine, case.names), case.key, case.off, case.ids, case.score, thr, dis, correct)
    (cell, cnt, off, ids, dropped), n = case.expected(thr, dis, correct)
    msg = (case.name, thr, dis, correct)
    assert np.array_equal(cell, t.cell) and np.array_equal(cnt, t.count), msg
    assert np.array_equal(off.astype(np.int64), t.feat_off.astype(np.int64)) and np.array_equal(ids, t.feat_ids), msg
    assert dropped == t.dropped_empty, msg
    if correct:
        assert t.umis_corrected == n, msg
    return t


def run(engine, case, correct=(False, True)):
    """every threshold of the case, then thresholding off; with and without correction where the case has UMI strings"""
    for c in correct:
        if c and case.umis is None:
            continue
        for thr in case.thresholds:
            check(engine, case, thr, False, c)
        check(engine, case, case.thresholds[0], True, c)


def _write_tsv(path, rows):
    with open(path, "w") as f:
        f.write("nimble_features\tnimble_score\tr1_CB\tr1_UB\n")
        f.write("".join("%s\t%r\t%s\t%s\n" % (feats, score, cb, umi) for cb, umi, feats, score in rows))


def tsv_route(engine, tmp_path, case, thr, dis, correct):
    """per-read TSV -> nb200_report_file -> bytes of report_counts on the (corrected) rows"""
    tsv, got = str(tmp_path / "in.tsv"), str(tmp_path / "out.tsv")
    _write_tsv(tsv, case.rows)
    fixed, n = correct_umis(case.rows) if correct else (case.rows, None)
    out, dropped = report_counts(fixed, thr, dis)
    o = engine.report_file(tsv, got, thr, dis, correct)
    assert o[1:3] == (len(out), dropped), (case.name, thr, dis, correct)
    if correct:
        assert o[3] == n
    with open(got, "rb") as f:
        assert f.read() == "".join("%s\t%d\t%s\n" % r for r in out).encode(), (case.name, thr, dis, correct)


# ---- 1. token packing ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("F", [127, 128, 511, 512, 32767, 32768, 200_000])
def test_token_packing(engine, F):
    names = U.hla_names(F)
    for nf in U.token_max_nf(F):
        for big in (False, True):
            c = U.token_case(F, nf, big, names=names)
            if F > 100_000:
                c.thresholds = (0.05,)
            run(engine, c, (False,))
            check(engine, c, 0.05, False, True)


# ---- 2. group sort -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [48, 49])
def test_group_sort(engine, tmp_path, n):
    c = U.group_sort_case(n)
    run(engine, c)
    thr = c.thresholds[0]
    for correct in (False, True):
        tsv_route(engine, tmp_path, c, thr, False, correct)


# ---- 3. general-kernel working set ---------------------------------------------------------------------------------
def test_general_working_set(engine, tmp_path):
    c = U.general_case()
    run(engine, c)
    tsv_route(engine, tmp_path, c, 0.05, False, True)


# ---- 4. stage-2 key width ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C,D", [(1 << 15, 1 << 16), (1 << 15, (1 << 16) + 1), ((1 << 20) + 1, (1 << 17) + 1),
                                 (1, 1 << 16), (1, (1 << 16) + 1)])
def test_stage2_key_width(engine, C, D):
    c = U.stage2_case(C, D)
    if c.umis is None:
        check(engine, c, 0.3, False)
    else:
        run(engine, c, (False,))
        check(engine, c, 0.3, False, True)


# ---- 5. count width and cells --------------------------------------------------------------------------------------
def test_count_width_and_cell_rows(engine):
    c = U.count_width_case()
    t = check(engine, c, 0.05, False)
    assert set(t.count[t.cell == 7].tolist()) == {255, 256, 70000} and int((t.cell == 9).sum()) == 66000
    check(engine, c, 0.05, True)


# ---- 6. keys -------------------------------------------------------------------------------------------------------
def test_key_bits(engine):
    run(engine, U.keys_case(), (False,))


def test_four_million_distinct_keys(engine):
    c = U.many_keys_case()
    t = check(engine, c, 0.05, False)
    assert t.n_umis == len(c.key)


# ---- 7. float edges ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("make", [U.float_edges_case, U.knife_simple_case, U.knife_general_case, U.kahan_small_case],
                         ids=["float_edges", "knife_simple", "knife_general", "kahan_small"])
def test_float_edges(engine, make):
    run(engine, make())


# ---- 8. correction -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("make", [U.grow_past_48_case, U.big_umi_case, U.one_base_case, U.thirteen_case, U.ties_case],
                         ids=["grow_past_48", "big_umi", "one_base", "thirteen", "ties"])
def test_correction(engine, tmp_path, make):
    c = make()
    run(engine, c)
    for dis in (False, True):
        tsv_route(engine, tmp_path, c, 0.05, dis, True)


@pytest.mark.parametrize("m", U.SELECTED_M)
def test_correction_selected_rows(engine, m):
    c = U.selected_rows_case(m)
    t = check(engine, c, 0.05, False, True)
    assert t.n_called == m
    check(engine, c, 0.05, True, True)
    check(engine, c, 0.05, False)


# ---- 9. file route, correction, two libraries ----------------------------------------------------------------------
def _per_read_rows(path):
    with open(path) as f:
        head = f.readline().rstrip("\n").split("\t")
        fi, si, ci, ui = (head.index(h) for h in ("nimble_features", "nimble_score", "r1_CB", "r1_UB"))
        rows = []
        for line in f:
            r = line.rstrip("\n").split("\t")
            rows.append((r[ci], r[ui], r[fi], float(r[si]) if r[si] else float("nan")))
    return rows


def test_file_route_two_libraries(engine, tmp_path):
    """one align_files_counts call over two libraries, a UMI whose group passes 48 rows only after correction: equal,
    per library, to align then report_file, and to the string oracles"""
    import file_bench
    lib_a, codes = synth.allele_family_library(n_founders=6, alleles_per_founder=12, length=600, snps_mean=10, seed=91)
    lib_b, _ = synth.allele_family_library(n_founders=6, alleles_per_founder=12, length=600, snps_mean=10, seed=91,
                                           name_prefix="Other")
    lib_b[1]["columns"] = [col[: len(col) // 2] for col in lib_b[1]["columns"]]     # half the references
    paths = []
    for i, lib in enumerate((lib_a, lib_b)):
        paths.append(str(tmp_path / ("lib%d.json" % i)))
        with open(paths[-1], "w") as f:
            json.dump(lib, f)
    r1, truth = synth.sample_reads(codes, 30_000, read_len=90, seed=92)
    key = synth.barcodes_10x(len(r1), n_cells=100, seed=93, truth=truth)
    blk, _ = synth.sample_reads(codes, 58, read_len=90, err_rate=0.0, off_target=0.0, n_frac=0.0, seed=94, ref_idx=np.arange(58) % 4)
    u = 0x5A5A5A                                           # 12-base UB, 2 bits a base; v = u with one base changed
    v = u ^ (2 << 10)
    bkey = np.array([(0xC0FFEE01 << 32) | (u if i < 48 else v) for i in range(58)], np.uint64)
    r1 = np.concatenate([r1, blk])
    key = np.concatenate([key, bkey])
    bam = str(tmp_path / "in.bam")
    file_bench.write_bam(bam, r1, key)
    la, lb = engine.load_library(paths[0]), engine.load_library(paths[1])
    per = [str(tmp_path / "a.tsv"), str(tmp_path / "b.tsv")]
    engine.align_files([bam], [la, lb], per)
    rows_a = _per_read_rows(per[0])                       # input order: the block is last
    cell = rows_a[-1][0]

    def largest(rows):
        n = {}
        for cb, umi, feats, score in rows:
            if cb == cell and umi and feats and score == score:
                n[umi] = n.get(umi, 0) + 1
        return max(n.values())
    assert largest(rows_a) <= U.LOCAL_SORT_MAX < largest(correct_umis(rows_a)[0])
    for thr, dis in ((0.05, False), (0.05, True)):
        got = [str(tmp_path / "got_a.tsv"), str(tmp_path / "got_b.tsv")]
        o = engine.align_files_counts([bam], [la, lb], got, None, thr, dis, True)
        for i in range(2):
            want = str(tmp_path / ("want%d.tsv" % i))
            assert o[i] == engine.report_file(per[i], want, thr, dis, True), (i, thr, dis)
            with open(want, "rb") as f:
                w = f.read()
            with open(got[i], "rb") as f:
                assert f.read() == w, (i, thr, dis)
            fx, n = correct_umis(_per_read_rows(per[i]))
            out, dropped = report_counts(fx, thr, dis)
            assert w == "".join("%s\t%d\t%s\n" % r for r in out).encode() and o[i][2:] == (dropped, n), (i, thr, dis)
    assert o[0][3] != o[1][3] or o[0][1] != o[1][1]           # the libraries see different rows


# ---- 10. seeded sweep ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", range(7000, 7000 + int(os.environ.get("NB200_FUZZ_CASES", "12"))))
def test_sweep(engine, seed):
    c = U.sweep_case(seed)
    run(engine, c)
