#!/usr/bin/env python
"""Raw 10x FASTQ routes of this tree against another build: `fastq-to-bam` and `align --map`, wall clock and peak RSS.

    python scripts/tenx_stream_bench.py --baseline DIR [--sizes 4000000,24000000] [--runs 3] [--out-dir /tmp/nb200_tenx]

DIR is a built checkout of another revision (its nimble_b200/libnimble_b200.so in place).  For each size the script
writes seeded plain-gzip R1 / R2 (R1 = 16 + 12 + 62 bases, R2 = 90, 737 k-entry whitelist: scripts/file_bench.py --tenx)
from a child process, then runs each route from both builds, alternating which goes first, each in a process of its
own, `--runs` times.  The decompressed BAM streams, the per-read TSVs and the printed counters of the two builds must be
identical (exit code 4 otherwise).  `align --map` of this tree also runs on 2 GPUs, and on 8 where the node has them,
and must write the same TSV.  Prints one JSON line; the card's name and power limit are read in the same run.

A long size may not fit one process's time budget: `--runs 1 --run0 R --merge PREV.json` runs one more alternating run and
prints PREV's runs and this one as one result (same sizes, same card, same seeded input; identity is required of every
run merged)."""
import argparse
import gzip
import hashlib
import json
import os
import re
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "scripts"))
sys.path.insert(0, ROOT)
import file_bench  # noqa: E402
from nimble_b200 import synth  # noqa: E402


def run(tree, argv):
    """`python -m nimble_b200 argv` from the tree `tree`: (wall seconds, peak RSS MB, rc, stdout)."""
    t0 = time.perf_counter()
    p = subprocess.Popen([sys.executable, "-m", "nimble_b200"] + argv, cwd=tree, stdout=subprocess.PIPE, text=True,
                         env=dict(os.environ, PYTHONPATH=tree))
    out = p.stdout.read()
    _, status, ru = os.wait4(p.pid, 0)
    return time.perf_counter() - t0, ru.ru_maxrss / 1024.0, os.waitstatus_to_exitcode(status), out


def digest(path, gz=False):
    h = hashlib.sha256()
    with (gzip.open(path, "rb") if gz else open(path, "rb")) as f:
        for b in iter(lambda: f.read(1 << 24), b""):
            h.update(b)
    return h.hexdigest()


def counters(stdout):
    """The counter lines of fastq-to-bam's report / align --map's summary line (timings left out)."""
    keep = [l for l in stdout.splitlines() if re.search(r"pairs|matches|Corrected|correction|mismatch|short|remaining|cache size", l)]
    return [re.sub(r" -> .*", "", l) for l in keep]


def median(v):
    v = sorted(v)
    return v[len(v) // 2]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline", required=True, help="a built checkout of the revision to compare with")
    ap.add_argument("--sizes", default="4000000,24000000")
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--run0", type=int, default=0, help="index of the first run (run r starts with this tree when r is even): "
                                                        "lets several calls, e.g. one run each, continue the alternation")
    ap.add_argument("--baseline-label", default=None, help="what the baseline is, for the JSON (default: its directory name)")
    ap.add_argument("--merge", default=None, help="the JSON printed by an earlier call: its runs are added to this one's")
    ap.add_argument("--cores", type=int, default=0)
    ap.add_argument("--out-dir", default="/tmp/nb200_tenx_stream_bench")
    args = ap.parse_args()
    base = os.path.abspath(args.baseline)
    os.makedirs(args.out_dir, exist_ok=True)
    cores = str(args.cores or os.cpu_count())
    import torch
    n_gpus = torch.cuda.device_count()
    lib, _ = synth.allele_family_library(n_founders=40, alleles_per_founder=50, length=1098, snps_mean=15.0, seed=1)
    lib_path = os.path.join(args.out_dir, "lib.json")
    with open(lib_path, "w") as f:
        json.dump(lib, f)
    res = {"host_threads": int(cores), "gpus_on_node": n_gpus, "input": "plain gzip (one zlib stream per file)",
           "whitelist": 737_280, "baseline": args.baseline_label or os.path.basename(base.rstrip("/")), "sizes": {}}
    res.update(file_bench.gpu_info())
    prev = None
    if args.merge:
        with open(args.merge) as f:
            prev = json.load(f)
        for k in ("host_threads", "gpu_name", "gpu_power_limit", "baseline"):
            if prev.get(k) != res.get(k):
                sys.exit("--merge: %s differs (%r against %r)" % (k, prev.get(k), res.get(k)))
    ok = True
    for n in [int(x) for x in args.sizes.split(",")]:
        d = os.path.join(args.out_dir, "p%d" % n)
        os.makedirs(d, exist_ok=True)
        t0 = time.time()
        import multiprocessing                       # (a child process: the timed routes must not inherit its peak RSS)
        p = multiprocessing.get_context("spawn").Process(target=file_bench._write_tenx_child, args=(d, n))
        p.start(); p.join()
        if p.exitcode != 0:
            sys.exit("writing the 10x FASTQs failed")
        r1, r2, wl = (os.path.join(d, f) for f in ("R1.fastq.gz", "R2.fastq.gz", "whitelist.txt"))
        print("%d pairs written in %.0f s" % (n, time.time() - t0), file=sys.stderr)
        row = {k: {"new": [], "base": []} for k in ("fastq_to_bam_s", "fastq_to_bam_rss_mb", "align_map_s", "align_map_rss_mb")}
        seen = {}
        for r in range(args.run0, args.run0 + args.runs):
            for who, tree in ((("new", ROOT), ("base", base)) if r % 2 == 0 else (("base", base), ("new", ROOT))):
                bam, tsv = os.path.join(d, "%s.bam" % who), os.path.join(d, "%s.tsv" % who)
                a = run(tree, ["fastq-to-bam", "--r1-fastq", r1, "--r2-fastq", r2, "--map", wl, "--output", bam, "-c", cores])
                b = run(tree, ["align", "--reference", lib_path, "--input", r1, r2, "--map", wl, "--output", tsv, "-c", cores])
                if a[2] or b[2]:
                    sys.exit("%s build failed at %d pairs: rc %d / %d" % (who, n, a[2], b[2]))
                row["fastq_to_bam_s"][who].append(a[0]); row["fastq_to_bam_rss_mb"][who].append(a[1])
                row["align_map_s"][who].append(b[0]); row["align_map_rss_mb"][who].append(b[1])
                if r == args.run0:
                    seen[who] = (digest(bam, gz=True), digest(tsv), counters(a[3]), counters(b[3]))
        same = seen["new"] == seen["base"]
        old = (prev or {}).get("sizes", {}).get(str(n))
        if old:                                      # an earlier call's runs of this size: same input, same outputs
            for k in ("fastq_to_bam_s", "fastq_to_bam_rss_mb", "align_map_s", "align_map_rss_mb"):
                for w in ("new", "base"):
                    row[k][w] = old[k][w] + row[k][w]
            same = same and old["identical_bam_tsv_counters"] and old["counters"] == seen["new"][2] + seen["new"][3]
        multi = {}
        for g in [x for x in (2, 8) if x <= n_gpus]:
            tsv = os.path.join(d, "new_%dgpu.tsv" % g)
            c = run(ROOT, ["align", "--reference", lib_path, "--input", r1, r2, "--map", wl, "--output", tsv, "-c", cores, "--gpus", str(g)])
            multi[str(g)] = {"align_map_s": c[0], "align_map_rss_mb": c[1], "tsv_identical": c[2] == 0 and digest(tsv) == seen["new"][1]}
            ok &= multi[str(g)]["tsv_identical"]
        if old:
            multi = dict(old["multi_gpu"], **multi)
        row.update(runs=len(row["fastq_to_bam_s"]["new"]), identical_bam_tsv_counters=same, counters=seen["new"][2] + seen["new"][3], multi_gpu=multi,
                   median_new_over_base={k: median(v["new"]) / median(v["base"]) for k, v in row.items() if isinstance(v, dict) and "new" in v})
        res["sizes"][str(n)] = row
        ok &= same
        for f in os.listdir(d):                      # (tens of GB at 24 M pairs)
            if f.endswith((".bam", ".tsv")):
                os.remove(os.path.join(d, f))
    if prev:                                         # sizes only the earlier call ran
        for k, v in prev["sizes"].items():
            res["sizes"].setdefault(k, v)
    print(json.dumps(res))
    if not ok:
        sys.exit(4)


if __name__ == "__main__":
    main()
