"""The slab re-run of the streaming file pipeline (lane_wait): a slab whose Smith-Waterman work list overflows is run again
with a larger list.  A child process whose work list starts at 64 items (NB200_ITEMS_CAP) re-runs slabs; its outputs must
be the bytes of a normal run, so a re-run appends its rows anew and logs its barcodes again without changing anything."""
import json
import os
import subprocess
import sys

import pytest

from nimble_b200 import synth
from test_fastq_counts_gpu import KEYS, _library, _tenx

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "scripts"))

pytestmark = pytest.mark.gpu

CHILD = r'''
import json, sys
sys.path.insert(0, %r)
import nimble_b200
method, lib_paths, args = json.loads(sys.argv[1])
eng = nimble_b200.Engine(0)
libs = [eng.load_library(p) for p in lib_paths]
out = getattr(eng, method)(*[libs if a == "LIBS" else a for a in args])
print("RESULT " + json.dumps(out))
''' % ROOT


def _capped(method, lib_paths, args):
    """Engine.<method>(*args) on a fresh engine in a child process whose work list starts at 64 items; "LIBS" in args
    stands for the libraries loaded from lib_paths.  Returns the call's result as JSON would carry it."""
    env = dict(os.environ, NB200_ITEMS_CAP="64")
    out = subprocess.run([sys.executable, "-c", CHILD, json.dumps([method, lib_paths, args])], env=env, capture_output=True,
                         text=True, timeout=600)
    assert out.returncode == 0, out.stdout + out.stderr
    return json.loads(out.stdout.split("RESULT ", 1)[1])


def _read(p):
    with open(p, "rb") as f:
        return f.read()


@pytest.fixture(scope="module")
def bam_input(tmp_path_factory):
    """300 k single-end reads (three slabs) with 2 % substitutions, so that every slab has Smith-Waterman work."""
    import file_bench
    tmp_path = tmp_path_factory.mktemp("swretry")
    lib_path, codes = _library(tmp_path, 81)
    r1, truth = synth.sample_reads(codes, 300_000, read_len=90, err_rate=0.02, seed=82)
    key = synth.barcodes_10x(len(r1), n_cells=500, seed=82, truth=truth)
    bam = str(tmp_path / "in.bam")
    file_bench.write_bam(bam, r1, key)
    return tmp_path, lib_path, bam


def test_align_files_rerun(engine, bam_input):
    tmp_path, lib_path, bam = bam_input
    want, got = str(tmp_path / "a_want.tsv"), str(tmp_path / "a_got.tsv")
    engine.align_files([bam], [engine.load_library(lib_path)], [want])
    _capped("align_files", [lib_path], [[bam], "LIBS", [got]])
    assert _read(got) == _read(want) and len(_read(want)) > 1_000_000


def test_align_files_counts_rerun(engine, bam_input):
    tmp_path, lib_path, bam = bam_input
    want, got = str(tmp_path / "c_want.tsv"), str(tmp_path / "c_got.tsv")
    o3_want = engine.align_files_counts([bam], [engine.load_library(lib_path)], [want])
    o3_got = _capped("align_files_counts", [lib_path], [[bam], "LIBS", [got]])
    assert o3_got == json.loads(json.dumps(o3_want)) and o3_want[0][0] > 100_000
    assert _read(got) == _read(want)


def test_fastq_to_counts_rerun(engine, tmp_path):
    """300 k pairs (three slabs): counts, out3 and the barcode statistics."""
    lib_path, codes = _library(tmp_path, 91)
    f1, f2, wlp, _, _, _ = _tenx(tmp_path, codes, 300_000, 92)
    want, got = str(tmp_path / "t_want.tsv"), str(tmp_path / "t_got.tsv")
    st_want, o3_want = engine.fastq_to_counts(f1, f2, wlp, [engine.load_library(lib_path)], [want])
    st_got, o3_got = _capped("fastq_to_counts", [lib_path], [f1, f2, wlp, "LIBS", [got]])
    assert o3_got == json.loads(json.dumps(o3_want))
    for k in KEYS + ("n_exact_miss", "n_multi"):
        assert st_got[k] == st_want[k], k
    assert o3_want[0][0] > 100_000 and st_want["n_multi"] > 0
    assert _read(got) == _read(want)
