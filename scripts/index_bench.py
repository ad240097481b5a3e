#!/usr/bin/env python
"""Start-up cost of a library: `align --counts` from the library JSON (index built in the call) against the same call
from an index file written once by `index`.  Every measurement is its own `python -m nimble_b200` process, the two
routes alternate, and the counts files of the two routes must be identical.  Records wall clock, peak RSS, the card's
name and power limit, and the per-library load trace (NB200_TRACE: host time, image copy, device checksum).

    python scripts/index_bench.py [--workload cfg2|cfg5] [--transcripts 25000] [--gpus 1,8] [--reads 200000] [--repeats 3]
"""
import argparse
import filecmp
import json
import os
import re
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
from nimble_b200 import synth  # noqa: E402


def gpu_info():
    """Card name, power limit and max SM clock (read-only nvidia-smi query): part of every number this script prints."""
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True,
                         text=True, timeout=30).stdout.strip().splitlines()
    return {"nvidia_smi": out[:2], "gpu_count": len(out) - 1}


def run(argv, env=None):
    """One process: (wall seconds, peak RSS MB, rc, stderr)."""
    t0 = time.perf_counter()
    p = subprocess.Popen([sys.executable, "-m", "nimble_b200"] + argv, cwd=ROOT, stdout=subprocess.DEVNULL, stderr=subprocess.PIPE,
                         text=True, env=env)
    err = p.stderr.read()
    _, status, ru = os.wait4(p.pid, 0)
    return time.perf_counter() - t0, ru.ru_maxrss / 1024.0, os.waitstatus_to_exitcode(status), err


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg5"])
    ap.add_argument("--transcripts", type=int, default=25000, help="cfg5: synthetic transcripts (200000 = full scale)")
    ap.add_argument("--gpus", default="1", help="comma-separated GPU counts to run (e.g. 1,8)")
    ap.add_argument("--reads", type=int, default=200000, help="reads of the (small) BAM: the call is dominated by start-up")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--cores", type=int, default=16)
    ap.add_argument("--out", default=None, help="JSON result path (default: stdout only)")
    args = ap.parse_args()
    import file_bench
    tmp = tempfile.mkdtemp(prefix="nb200_index_bench_")
    if args.workload == "cfg5":
        lib, codes = synth.random_transcript_library(n_seqs=args.transcripts, mean_len=2000, family_frac=0.3, seed=5,
                                                     config={"score_percent": 0.25})
        k, rl = 31, 100
    else:
        lib, codes = synth.allele_family_library(n_founders=40, alleles_per_founder=50, length=1098, snps_mean=15.0, seed=1)
        k, rl = 20, 90
    js, idx, bam = os.path.join(tmp, "lib.json"), os.path.join(tmp, "lib.nb200idx"), os.path.join(tmp, "in.bam")
    with open(js, "w") as f:
        json.dump(lib, f)
    del lib
    r1, truth = synth.sample_reads(codes, args.reads, read_len=rl, seed=7)
    key = synth.barcodes_10x(args.reads, n_cells=2000, seed=7, truth=truth)
    file_bench.write_bam(bam, r1, key)
    out = {"workload": args.workload, "transcripts": args.transcripts if args.workload == "cfg5" else None, "k": k,
           "reads": args.reads, "host_threads": args.cores}
    out.update(gpu_info())
    w = run(["index", "--reference", js, "--output", idx, "-k", str(k), "-c", str(args.cores)])
    assert w[2] == 0, w[3]
    out.update(index_write_s=w[0], index_write_rss_mb=w[1], index_bytes=os.path.getsize(idx), json_bytes=os.path.getsize(js))
    env = dict(os.environ, NB200_TRACE="1")
    trace = re.compile(r"\[nb200 trace\] library .*")
    for g in [int(x) for x in args.gpus.split(",")]:
        if g > out["gpu_count"]:
            out["gpus_%d" % g] = "skipped: %d GPUs on this node" % out["gpu_count"]
            continue
        res = {"json_s": [], "json_rss_mb": [], "index_s": [], "index_rss_mb": [], "trace_json": [], "trace_index": []}
        cnt = {}
        for rep in range(args.repeats + 1):                      # repetition 0 warms the page cache and the driver
            for route, ref in (("json", js), ("index", idx)):
                cnt[route] = os.path.join(tmp, "counts_%s_%d.tsv" % (route, g))
                t, rss, rc, err = run(["align", "--reference", ref, "--input", bam, "--counts", cnt[route], "-k", str(k),
                                       "-c", str(args.cores), "--gpus", str(g)], env)
                assert rc == 0, err[-2000:]
                if rep:
                    res[route + "_s"].append(t); res[route + "_rss_mb"].append(rss)
                    res["trace_" + route] += trace.findall(err)
        res["counts_identical"] = filecmp.cmp(cnt["json"], cnt["index"], shallow=False)
        res["saving_s"] = min(res["json_s"]) - min(res["index_s"])
        out["gpus_%d" % g] = res
        if not res["counts_identical"]:
            print(json.dumps(out))
            sys.exit(4)
    print(json.dumps(out))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
