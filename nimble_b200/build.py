"""Builds nimble_b200/libnimble_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libnimble_b200.so")
SOURCES = ["engine.cu", "library.cpp", "ingest.cpp", "stream.cpp", "fastq2bam.cpp", "report.cpp"]
ALIGNER = os.path.join(HERE, "aligner")
HEADERS = ["kernels.cuh", "agg.cuh", "barcode.cuh", "library.hpp", "json.hpp", "ingest.hpp", "kmer_hash.hpp", "checksum.hpp", "stream.hpp", "slab_api.hpp", "trim.hpp", "fast_inflate.hpp", "pandas_na.hpp", "umi_code.hpp", "aligner_main.cpp", os.path.join("..", "..", "include", "nimble_b200.h")]


def nvcc_path():
    for p in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if p and os.path.exists(p):
            return p
    raise RuntimeError("nvcc not found")


def needs_build():
    if not os.path.exists(OUT) or not os.path.exists(ALIGNER):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(os.path.join(CSRC, f)) > t for f in SOURCES + HEADERS)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return OUT
    cmd = [nvcc_path(), "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
           "-fmad=false", "-Xcompiler", "-fPIC,-O3,-Wall", "-shared", "-ccbin", "/usr/bin/g++",
           "-Xptxas", "-v" if verbose else "-O3", "-o", OUT] + [os.path.join(CSRC, s) for s in SOURCES] + ["-lz"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed")
    if verbose:
        print(r.stdout + r.stderr)
    # the `aligner` executable nimble's unmodified front end execs (nimble/__main__.py:154,195)
    r = subprocess.run(["/usr/bin/g++", "-O2", "-std=c++17", "-o", ALIGNER, os.path.join(CSRC, "aligner_main.cpp"),
                        "-I", os.path.join(HERE, "..", "include"), "-L", HERE, "-lnimble_b200", "-Wl,-rpath,$ORIGIN"],
                       capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("aligner link failed")
    return OUT


if __name__ == "__main__":
    build(force=True, verbose="-v" in sys.argv)
    print("built", OUT)
