"""An engine returns every device allocation it made when it is closed, including the state of a call that failed.  Ten
create / use / close cycles in one process run the resident path, both counts routes, barcode correction and a
fastq-to-counts call that fails after its slabs are on the device; the process's GPU memory must stay flat after the
first two cycles (which load the kernel modules)."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import nimble_b200
from nimble_b200 import synth
from nimble_b200._lib import NimbleB200Error
from test_fastq_counts_gpu import _library, _tenx, _write_fastq

pytestmark = pytest.mark.gpu

CYCLES = 10


def _gpu_mib():
    """This process's GPU memory in MiB as nvidia-smi lists it (read-only query), or None where it does not list it."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-compute-apps=pid,used_memory", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=60)
    except (OSError, subprocess.TimeoutExpired):
        return None
    if out.returncode != 0:
        return None
    total, seen = 0, False
    for line in out.stdout.splitlines():
        parts = [p.strip() for p in line.split(",")]
        if len(parts) == 2 and parts[0] == str(os.getpid()) and parts[1].isdigit():
            total += int(parts[1])
            seen = True
    return total if seen else None


@pytest.fixture(scope="module")
def inputs(tmp_path_factory):
    import file_bench
    tmp = tmp_path_factory.mktemp("lifetime")
    lib_path, codes = _library(tmp, 81)
    r1, truth = synth.sample_reads(codes, 20_000, read_len=90, seed=82)
    key = synth.barcodes_10x(len(r1), n_cells=200, seed=82, truth=truth)
    bam = str(tmp / "in.bam")
    file_bench.write_bam(bam, r1, key)
    f1, f2, wlp, wl, cb, q = _tenx(tmp, codes, 5_000, 83)
    # a pair whose barcode is corrected and whose name is over 254 bytes: fails in the slab's wait, after its upload
    r2b, _ = synth.sample_reads(codes, 200, read_len=90, seed=84)
    recs = [("g%d" % i, wl[0] + "ACGTTGCAACGT" + "ACGT" * 15, r2b[i].tobytes().decode()) for i in range(200)]
    recs.insert(100, ("n" * 300, wl[0] + "ACGTTGCAACGT" + "ACGT" * 15, r2b[0].tobytes().decode()))
    b1, b2 = str(tmp / "bad_1.fastq"), str(tmp / "bad_2.fastq")
    _write_fastq(b1, [(n, a, "F" * len(a)) for n, a, _ in recs])
    _write_fastq(b2, [(n, b, "F" * len(b)) for n, _, b in recs])
    return tmp, lib_path, r1, key, bam, (f1, f2, wlp), wl, cb, q, (b1, b2)


def _cycle(inputs):
    tmp, lib_path, r1, key, bam, (f1, f2, wlp), wl_lines, cb, q, (b1, b2) = inputs
    eng = nimble_b200.Engine(0)
    try:
        lib = eng.load_library(lib_path)
        table = eng.align(lib, r1, key=key)
        assert len(table) > 0 and len(eng.align_resident(lib)) == len(table)
        assert eng.align_files_counts([bam], [lib], [str(tmp / "a.tsv")])[0][0] > 0
        st, o3 = eng.fastq_to_counts(f1, f2, wlp, [lib], [str(tmp / "f.tsv")])
        assert st["written_pairs"] > 0 and o3[0][0] > 0
        wl = eng.load_whitelist(wl_lines)
        idx, _, _ = eng.correct_barcodes(wl, cb, q)
        assert (idx >= 0).any()
        with pytest.raises(NimbleB200Error, match="254 bytes"):
            eng.fastq_to_counts(b1, b2, wlp, [lib], [str(tmp / "bad.tsv")])
    finally:
        eng.close()


def test_create_use_close_returns_device_memory(inputs):
    mib = []
    for _ in range(CYCLES):
        _cycle(inputs)
        m = _gpu_mib()
        if m is None:
            pytest.skip("nvidia-smi --query-compute-apps is unavailable or does not list this process")
        mib.append(m)
    assert max(mib[2:]) <= mib[1], "GPU memory after each create / use / close cycle (MiB): %s" % mib
