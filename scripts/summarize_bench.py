#!/usr/bin/env python
"""`report -s` native (nb200_summarize_file: host parse and write, grouping on the GPU) against the Python path
(frontend.summarize_fields_tsv).  Seeded per-read TSVs of align's 13 columns, `-s r1_GN,r1_POS,nimble_features`, at
12 M and 50 M rows (the Python path at 12 M only: it holds every row as Python strings).  Every run is a process of its
own, the two paths alternate, and each reports its wall clock (from before the engine is created to the file written),
its peak RSS and, for the native path, CUDA-event times from nb200_last_timing: device_kernel_ms (agg_ms) is the kernels
and sorts of the grouping; device_total_ms (total_ms) spans the first upload to the last download, so it also holds the
host work that builds each column's rows between them.  The outputs must be byte-identical.  The card's name and
power limit are read in the same call.

    python scripts/summarize_bench.py [--rows 12000000,50000000] [--repeats 2] [--python-repeats 1] [--out profiles/r03_summarize_bench_1gpu.json]
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COLUMNS = ["nimble_features", "nimble_score", "r1_forward_score", "r1_reverse_score", "r2_forward_score", "r2_reverse_score",
           "r1_QNAME", "r1_CB", "r1_UB", "r1_UR", "r1_GN", "r1_POS", "r2_POS"]
SUMMARIZE = ["r1_GN", "r1_POS", "nimble_features"]

CHILD = r"""
import json, os, resource, sys, time
sys.path.insert(0, %(root)r)
mode, inp, out = sys.argv[1:4]
cols = sys.argv[4].split(",")
t0 = time.perf_counter()
res = {}
if mode == "native":
    from nimble_b200 import Engine
    eng = Engine(0)
    rows, umis = eng.summarize_file(inp, cols, out)
    tm = eng.timing()
    res.update(rows=rows, umis=umis, device_total_ms=tm["total_ms"], device_kernel_ms=tm["agg_ms"], launches=tm["launches"])
    eng.close()
else:
    from nimble_b200 import frontend
    frontend.summarize_fields_tsv(inp, cols, out)
res["wall_s"] = time.perf_counter() - t0
res["peak_rss_gb"] = resource.getrusage(resource.RUSAGE_SELF).ru_maxrss / 1e6
print(json.dumps(res))
"""


def gpu_info():
    """Card name, power limit and max SM clock (read-only nvidia-smi query)."""
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                         text=True, timeout=30).stdout.strip().splitlines()
    return out[:2]


def write_tsv(path, n, seed=1):
    """align's per-read TSV shape: 5000 cells, 12-base UMIs drawn per read, 4 feature sets, 3 gene names (one blank)."""
    import numpy as np
    rng = np.random.default_rng(seed)
    cells = np.array(["".join(x) + "-1" for x in rng.choice(list("ACGT"), (5000, 16))])
    feats = np.array(["A", "B", "A,B", "C"])
    gn = np.array(["HLA-A", "HLA-B", ""])
    half = np.array(["".join("ACGT"[(c >> (2 * k)) & 3] for k in range(6)) for c in range(4096)])
    chunk = 1_000_000
    with open(path, "w") as f:
        f.write("\t".join(COLUMNS) + "\n")
        for a in range(0, n, chunk):
            m = min(chunk, n - a)
            umi = np.char.add(half[rng.integers(0, 4096, m)], half[rng.integers(0, 4096, m)])
            fe, cb, g = feats[rng.integers(0, 4, m)], cells[rng.integers(0, 5000, m)], gn[rng.integers(0, 3, m)]
            pos = rng.integers(1, 10 ** 8, m)
            f.write("".join("%s\t1\t90\t0\t0\t0\tread%d\t%s\t%s\t%s\t%s\t%d\t\n" % (fe[i], a + i, cb[i], umi[i], umi[i], g[i], pos[i])
                            for i in range(m)))


def run(mode, inp, out):
    r = subprocess.run([sys.executable, "-c", CHILD % {"root": ROOT}, mode, inp, out, ",".join(SUMMARIZE)], capture_output=True,
                       text=True)
    if r.returncode != 0:
        raise RuntimeError("%s run failed:\n%s" % (mode, r.stderr[-3000:]))
    res = json.loads(r.stdout.strip().splitlines()[-1])
    with open(out, "rb") as f:
        res["sha256"] = hashlib.sha256(f.read()).hexdigest()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", default="12000000,50000000")
    ap.add_argument("--python-rows", type=int, default=12_000_000, help="sizes at which the Python path also runs")
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--python-repeats", type=int, default=1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    report = {"workload": "per-read TSV, 13 columns, -s " + ",".join(SUMMARIZE), "gpu": gpu_info(), "sizes": []}
    with tempfile.TemporaryDirectory() as tmp:
        for n in [int(x) for x in a.rows.split(",")]:
            inp = os.path.join(tmp, "in.tsv")
            write_tsv(inp, n)
            entry = {"rows": n, "tsv_bytes": os.path.getsize(inp), "native": [], "python": []}
            py_left = a.python_repeats if n <= a.python_rows else 0
            for rep in range(a.repeats):
                entry["native"].append(run("native", inp, os.path.join(tmp, "native.tsv")))
                if py_left:
                    entry["python"].append(run("python", inp, os.path.join(tmp, "python.tsv")))
                    py_left -= 1
            hashes = {r["sha256"] for r in entry["native"] + entry["python"]}
            entry["outputs_identical"] = len(hashes) == 1
            for k in ("native", "python"):
                if entry[k]:
                    entry[k + "_best_wall_s"] = min(r["wall_s"] for r in entry[k])
                    entry[k + "_peak_rss_gb"] = max(r["peak_rss_gb"] for r in entry[k])
            print(json.dumps(entry), flush=True)
            report["sizes"].append(entry)
            os.unlink(inp)
    print(json.dumps(report))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(report, f, indent=1)
    if not all(e["outputs_identical"] for e in report["sizes"]):
        sys.exit(1)


if __name__ == "__main__":
    main()
