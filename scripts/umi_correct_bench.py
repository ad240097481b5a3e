#!/usr/bin/env python
"""Cost of UMI correction (NB200_UMI_CORRECT, DESIGN.md §2.12) in the UMI stage.  A cfg2-shaped report workload: 10 M rows
(synth.barcodes_10x: 10 000 cells, 3 reads per UMI), 12-base UMIs as their codes, 0.1 % per-base UMI errors, one feature
per molecule.  The rows go up once per call (nb200_umi_counts); the time is the stage's own (agg_ms, CUDA events from rows
resident to count table on the host).  The two settings alternate in one process, after one warm-up each; the card's name
and power limit are read in the same call.

    python scripts/umi_correct_bench.py [--rows 10000000] [--repeats 5] [--out profiles/r03_umi_correct_bench_cfg2_1gpu.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from nimble_b200 import Engine, synth  # noqa: E402


def gpu_info():
    """Card name, power limit and max SM clock (read-only nvidia-smi query)."""
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                         text=True, timeout=30).stdout.strip().splitlines()
    return out[:2]


def workload(n, err, seed=2):
    """key = cell << 32 | UMI code, CSR of one feature per row (the molecule's), the errors' rate per base."""
    key = synth.barcodes_10x(n, n_cells=10000, reads_per_umi=3.0, seed=seed)
    ub = key & np.uint64(0xFFFFFF)
    digits = np.stack([((ub >> np.uint64(2 * (11 - i))) & np.uint64(3)).astype(np.int64) for i in range(12)], axis=1)
    feat = (ub * np.uint64(2654435761) % np.uint64(1000)).astype(np.uint32)
    rng = np.random.default_rng(seed + 1)
    hit = rng.random(digits.shape) < err
    digits[hit] = (digits[hit] + rng.integers(1, 4, size=int(hit.sum()))) % 4        # another of A C G T
    code = np.zeros(n, np.uint64)
    for i in range(12):
        code = code * np.uint64(5) + (digits[:, i] + 1).astype(np.uint64)
    cell = np.unique(key >> np.uint64(32), return_inverse=True)[1].astype(np.uint64)
    return (cell << np.uint64(32)) | code, np.arange(n + 1, dtype=np.uint32), feat, int(hit.any(axis=1).sum())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=10_000_000)
    ap.add_argument("--err", type=float, default=0.001)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    key, off, feat, reads_with_error = workload(a.rows, a.err)
    eng = Engine(0)
    lib = eng.load_feature_names(["f%04d" % i for i in range(1000)])
    runs = {False: [], True: []}
    tables = {}
    for rep in range(a.repeats + 1):
        for corr in (False, True):
            t = eng.umi_counts(lib, key, off, feat, None, 0.05, False, corr)
            if rep:
                runs[corr].append(eng.timing()["agg_ms"])
            tables[corr] = t
    off_ms, on_ms = statistics.median(runs[False]), statistics.median(runs[True])
    res = {
        "what": "UMI stage (nb200_umi_counts agg_ms, rows resident) without and with NB200_UMI_CORRECT, alternating in one process",
        "gpu": gpu_info(),
        "rows": a.rows, "umi_bases": 12, "per_base_error": a.err, "rows_with_a_umi_error": reads_with_error,
        "agg_ms_off": runs[False], "agg_ms_on": runs[True],
        "median_ms_off": off_ms, "median_ms_on": on_ms, "added_ms": on_ms - off_ms,
        "umis_off": tables[False].n_umis, "umis_on": tables[True].n_umis, "umis_corrected": tables[True].umis_corrected,
        "count_rows_off": len(tables[False]), "count_rows_on": len(tables[True]),
        "counted_umis_off": int(tables[False].count.sum()), "counted_umis_on": int(tables[True].count.sum()),
    }
    eng.close()
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
