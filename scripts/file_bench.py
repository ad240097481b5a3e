#!/usr/bin/env python
"""File-level wall clock of the drop-in: synthetic 10x-like BAM (CB/UB tags) + library JSON ->
`align` (native BGZF reader, GPU path, per-read TSV) -> `report` (counts TSV).  Not the headline
metric (bench.py times the hot path); this is what a user of `python -m nimble_b200` waits for.

    python scripts/file_bench.py [--reads 2000000] [--out-dir /tmp/nb200_file_bench]
    python scripts/file_bench.py --tenx [--reads 20000000] [--gpus N]    # raw 10x FASTQ: fastq-to-bam + align --counts vs fastq-to-counts
"""
import argparse
import json
import os
import struct
import sys
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from nimble_b200 import frontend, synth  # noqa: E402


def bam_records(reads_ascii, key, id0=0):
    """Fixed-size unaligned single-end records (CB:Z 16-mer, UB:Z 12-mer) built with numpy; read names r<id0 + i>."""
    n, L = reads_ascii.shape
    name_len = 11
    rec = 32 + name_len + (L + 1) // 2 + L + 20 + 16
    a = np.zeros((n, 4 + rec), np.uint8)
    a[:, 0:4] = np.frombuffer(struct.pack("<i", rec), np.uint8)
    a[:, 4:36] = np.frombuffer(struct.pack("<iiBBHHHiiii", -1, -1, name_len, 0, 4680, 0, 4, L, -1, -1, 0), np.uint8)
    ids = np.arange(id0, id0 + n)
    a[:, 36] = ord("r")
    a[:, 37:46] = np.stack([(ids // 10 ** k) % 10 for k in range(8, -1, -1)], axis=1).astype(np.uint8) + ord("0")
    code = np.zeros(256, np.uint8)
    for ch, v in zip(b"ACGTN", (1, 2, 4, 8, 15)):
        code[ch] = v
    c = code[reads_ascii]
    if L % 2:
        c = np.concatenate([c, np.zeros((n, 1), np.uint8)], axis=1)
    o = 47
    a[:, o:o + c.shape[1] // 2] = (c[:, 0::2] << 4) | c[:, 1::2]
    o += c.shape[1] // 2
    a[:, o:o + L] = 30
    o += L
    acgt = np.frombuffer(b"ACGT", np.uint8)
    cb = (key >> np.uint64(32)).astype(np.uint64)
    ub = (key & np.uint64(0xFFFFFF)).astype(np.uint64)
    a[:, o:o + 3] = np.frombuffer(b"CBZ", np.uint8)
    a[:, o + 3:o + 19] = acgt[np.stack([(cb >> np.uint64(2 * (15 - j))) & np.uint64(3) for j in range(16)], axis=1).astype(np.int64)]
    o += 20
    a[:, o:o + 3] = np.frombuffer(b"UBZ", np.uint8)
    a[:, o + 3:o + 15] = acgt[np.stack([(ub >> np.uint64(2 * (11 - j))) & np.uint64(3) for j in range(12)], axis=1).astype(np.int64)]
    return a.tobytes()


def bgzf_append(f, raw, ex, level=1):
    """raw bytes -> 64 KB BGZF blocks appended to f (blocks need not end on record boundaries); returns bytes written."""
    view = memoryview(raw)

    def pack(span):                      # zlib releases the GIL: blocks are compressed on all host threads
        out = bytearray()
        for p in range(span[0], span[1], 0xFF00):
            blk = view[p:min(p + 0xFF00, span[1])]
            z = zlib.compressobj(level, zlib.DEFLATED, -15)
            cd = z.compress(blk) + z.flush()
            out += bytes([31, 139, 8, 4, 0, 0, 0, 0, 0, 255, 6, 0, 66, 67, 2, 0]) + struct.pack("<H", len(cd) + 25) + cd
            out += struct.pack("<II", zlib.crc32(blk), len(blk))
        return out

    step = 0xFF00 * 64
    total = 0
    for part in ex.map(pack, [(a, min(a + step, len(raw))) for a in range(0, len(raw), step)]):
        f.write(part)
        total += len(part)
    return total


BGZF_EOF = bytes([0x1F, 0x8B, 8, 4, 0, 0, 0, 0, 0, 0xFF, 6, 0, 0x42, 0x43, 2, 0, 0x1B, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0])


def write_bam(path, reads_ascii, key, level=1):
    """One call, everything in memory (small inputs)."""
    from concurrent.futures import ThreadPoolExecutor
    with open(path, "wb") as f, ThreadPoolExecutor(os.cpu_count() or 4) as ex:
        total = bgzf_append(f, b"BAM\x01" + struct.pack("<i", 0) + struct.pack("<i", 0) + bam_records(reads_ascii, key), ex, level)
        f.write(BGZF_EOF)
    return total + len(BGZF_EOF)


def write_bam_chunked(path, codes, n_reads, n_cells, chunk=4_000_000, seed=2, level=1):
    """Large inputs: reads are sampled, tagged and compressed chunk by chunk (memory stays at one chunk)."""
    from concurrent.futures import ThreadPoolExecutor
    total = 0
    with open(path, "wb") as f, ThreadPoolExecutor(os.cpu_count() or 4) as ex:
        total += bgzf_append(f, b"BAM\x01" + struct.pack("<i", 0) + struct.pack("<i", 0), ex, level)
        for c0 in range(0, n_reads, chunk):
            n = min(chunk, n_reads - c0)
            r1, truth = synth.sample_reads(codes, n, read_len=90, seed=seed + 7919 * (c0 // chunk))
            key = synth.barcodes_10x(n, n_cells=n_cells, seed=seed + 7919 * (c0 // chunk), truth=truth)
            total += bgzf_append(f, bam_records(r1, key, c0), ex, level)
        f.write(BGZF_EOF)
    return total + len(BGZF_EOF)


def gpu_info():
    """GPU name and power limit (read-only nvidia-smi query): part of every number this script prints."""
    import subprocess
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout
        first = out.strip().splitlines()[0].split(",")
        return {"gpu_name": first[0].strip(), "gpu_power_limit": first[1].strip()}
    except Exception as e:                      # noqa: BLE001 (recorded, not fatal)
        return {"gpu_info_error": str(e)}


def counts_bench(args, eng, kw, lib_path, bam, tsv, nbytes):
    """Two-step route (align -> per-read TSV -> report) against the fused `align --counts` (counts only), alternating
    them, two repetitions each; the counts files of the two routes must be byte-identical."""
    import filecmp
    two_counts, fused_counts = os.path.join(args.out_dir, "counts_two_step.tsv"), os.path.join(args.out_dir, "counts_fused.tsv")
    frontend.align(lib_path, tsv, [bam], args.cores, "unstranded", "", None, **kw)            # warm-up (CUDA context, page cache)
    frontend.align(lib_path, None, [bam], args.cores, "unstranded", "", None, counts=fused_counts, **kw)
    out = {"workload": args.workload, "reads": args.reads, "gpus": args.gpus, "host_threads": args.cores or os.cpu_count(),
           "bam_mb": nbytes / 1e6, "two_step_align_s": [], "two_step_report_s": [], "two_step_s": [], "fused_s": [], "rc": []}
    out.update(gpu_info())
    for _rep in range(2):
        os.remove(tsv)
        t0 = time.perf_counter()
        rc1 = frontend.align(lib_path, tsv, [bam], args.cores, "unstranded", "", None, **kw)
        t1 = time.perf_counter()
        frontend.report(tsv, two_counts, None, 0.05, False, engine=eng)
        t2 = time.perf_counter()
        rc2 = frontend.align(lib_path, None, [bam], args.cores, "unstranded", "", None, counts=fused_counts, **kw)
        t3 = time.perf_counter()
        out["two_step_align_s"].append(t1 - t0); out["two_step_report_s"].append(t2 - t1); out["two_step_s"].append(t2 - t0)
        out["fused_s"].append(t3 - t2); out["rc"] += [rc1, rc2]
    out["counts_identical"] = filecmp.cmp(two_counts, fused_counts, shallow=False)
    out["count_rows"] = sum(1 for _ in open(fused_counts))
    out["fused_reads_per_s"] = args.reads / min(out["fused_s"])
    print(json.dumps(out))
    if not out["counts_identical"] or any(out["rc"]):
        sys.exit(4)

def write_tenx_fastqs(out_dir, codes, n_pairs, chunk=2_000_000, seed=5, level=1):
    """Seeded raw 10x input: R1 = CB (synth.barcode_workload: 737 k-entry whitelist, errors, N, off-whitelist barcodes, 30 %
    clustered entries so that the correction cache decides) + UMI (12) + 62 bases, R2 = 90 bases, written as plain gzip
    (one member per chunk, not BGZF).  Returns (R1, R2, whitelist) paths."""
    from concurrent.futures import ThreadPoolExecutor
    r1p, r2p, wlp = (os.path.join(out_dir, f) for f in ("R1.fastq.gz", "R2.fastq.gz", "whitelist.txt"))
    wl_a = None
    acgt = np.frombuffer(b"ACGT", np.uint8)

    def fastq(ids, seq, qual, mate):                 # fixed-width names (p<9 digits>/<mate>): one numpy array per chunk
        n, L = seq.shape
        rec = np.zeros((n, 14 + 2 * L + 4), np.uint8)
        rec[:, 0] = ord("@"); rec[:, 1] = ord("p")
        rec[:, 2:11] = np.stack([(ids // 10 ** k) % 10 for k in range(8, -1, -1)], axis=1).astype(np.uint8) + ord("0")
        rec[:, 11] = ord("/"); rec[:, 12] = ord("0") + mate; rec[:, 13] = 10
        rec[:, 14:14 + L] = seq; rec[:, 14 + L] = 10; rec[:, 15 + L] = ord("+"); rec[:, 16 + L] = 10
        rec[:, 17 + L:17 + 2 * L] = qual; rec[:, -1] = 10
        return rec.tobytes()

    def gz(b):
        z = zlib.compressobj(level, zlib.DEFLATED, 31)
        return z.compress(b) + z.flush()

    with open(r1p, "wb") as f1, open(r2p, "wb") as f2, ThreadPoolExecutor(os.cpu_count() or 4) as ex:
        for c0 in range(0, n_pairs, chunk):
            n = min(chunk, n_pairs - c0)
            s = seed + 7919 * (c0 // chunk)
            rng = np.random.default_rng(s)
            if wl_a is None:                         # one whitelist and cell set; each chunk reads them in another order
                wl_a, cb0, q0 = synth.barcode_workload(chunk, n_whitelist=737_280, n_cells=10000, seed=seed, clustered=0.3)
            perm = rng.permutation(len(cb0))[:n]
            cb, q = cb0[perm], q0[perm]
            r2, _ = synth.sample_reads(codes, n, read_len=90, seed=s + 1)
            tail, _ = synth.sample_reads(codes, n, read_len=62, seed=s + 2)
            umi = acgt[rng.integers(0, 4, size=(n, 12))]
            s1 = np.concatenate([cb, umi, tail], axis=1)
            q1 = np.concatenate([q + 33, rng.integers(35, 75, size=(n, 74))], axis=1).astype(np.uint8)
            q2 = rng.integers(35, 75, size=(n, 90)).astype(np.uint8)
            ids = np.arange(c0, c0 + n)
            parts = list(ex.map(lambda a: gz(fastq(*a)), [(ids, s1, q1, 1), (ids, r2, q2, 2)]))
            f1.write(parts[0]); f2.write(parts[1])
    with open(wlp, "w") as f:
        f.write("\n".join(bytes(r).decode() for r in wl_a) + "\n")
    return r1p, r2p, wlp


def _write_tenx_child(out_dir, n_pairs):
    _, codes = synth.allele_family_library(n_founders=40, alleles_per_founder=50, length=1098, snps_mean=15.0, seed=1)
    write_tenx_fastqs(out_dir, codes, n_pairs)


def run_child(argv, env=None):
    """One `python -m nimble_b200 ...` process: (wall seconds, peak RSS MB, rc)."""
    import subprocess
    t0 = time.perf_counter()
    p = subprocess.Popen([sys.executable, "-m", "nimble_b200"] + argv, cwd=ROOT, stdout=subprocess.DEVNULL, env=env)
    _, status, ru = os.wait4(p.pid, 0)
    return time.perf_counter() - t0, ru.ru_maxrss / 1024.0, os.waitstatus_to_exitcode(status)


def tenx_bench(args, lib_path):
    """Raw 10x FASTQ to counts: `fastq-to-bam` then `align --counts` on its BAM (two processes, a BAM between them) against
    `fastq-to-counts` (one process, no BAM), alternating, two repetitions each.  Wall clock and peak RSS per process; the
    counts files must be byte-identical."""
    import filecmp
    t0 = time.time()
    made = {"tenx": args.reads}
    stamp = os.path.join(args.out_dir, "tenx.json")
    try:
        reuse = json.load(open(stamp)) == made
    except (OSError, ValueError):
        reuse = False
    r1p, r2p, wlp = (os.path.join(args.out_dir, f) for f in ("R1.fastq.gz", "R2.fastq.gz", "whitelist.txt"))
    if not reuse:
        # written by a child process: Linux keeps a process's peak RSS across fork + exec, so the routes timed below must
        # not be forked from a process that once held the generated data
        import multiprocessing
        p = multiprocessing.get_context("spawn").Process(target=_write_tenx_child, args=(args.out_dir, args.reads))
        p.start(); p.join()
        if p.exitcode != 0:
            sys.exit("writing the 10x FASTQs failed")
        with open(stamp, "w") as f:
            json.dump(made, f)
    print("%s 10x FASTQs: %d pairs, %.0f + %.0f MB in %.1fs" % ("reused" if reuse else "wrote", args.reads, os.path.getsize(r1p) / 1e6,
                                                              os.path.getsize(r2p) / 1e6, time.time() - t0), file=sys.stderr)
    cores = str(args.cores or os.cpu_count())
    bam, two, one = (os.path.join(args.out_dir, f) for f in ("tenx.bam", "tenx_counts_two_step.tsv", "tenx_counts_one_pass.tsv"))
    gp = ["--gpus", str(args.gpus)] if args.gpus > 1 else []
    step1 = ["fastq-to-bam", "--r1-fastq", r1p, "--r2-fastq", r2p, "--map", wlp, "--output", bam, "-c", cores]
    step2 = ["align", "--reference", lib_path, "--input", bam, "--counts", two, "-c", cores] + gp
    fused = ["fastq-to-counts", "--reference", lib_path, "--r1-fastq", r1p, "--r2-fastq", r2p, "--map", wlp, "--counts", one, "-c", cores] + gp
    out = {"pairs": args.reads, "gpus": args.gpus, "host_threads": int(cores), "r1_mb": os.path.getsize(r1p) / 1e6,
           "r2_mb": os.path.getsize(r2p) / 1e6, "whitelist": 737_280, "input": "plain gzip (one zlib stream per file)",
           "fastq_to_bam_s": [], "fastq_to_bam_rss_mb": [], "align_counts_s": [], "align_counts_rss_mb": [], "two_step_s": [],
           "one_pass_s": [], "one_pass_rss_mb": [], "rc": []}
    out.update(gpu_info())
    for _rep in range(2):
        a = run_child(step1)
        b = run_child(step2)
        c = run_child(fused, dict(os.environ, NB200_TRACE="1"))      # (stage times of the pipeline on stderr)
        out["fastq_to_bam_s"].append(a[0]); out["fastq_to_bam_rss_mb"].append(a[1])
        out["align_counts_s"].append(b[0]); out["align_counts_rss_mb"].append(b[1]); out["two_step_s"].append(a[0] + b[0])
        out["one_pass_s"].append(c[0]); out["one_pass_rss_mb"].append(c[1]); out["rc"] += [a[2], b[2], c[2]]
    out["counts_identical"] = filecmp.cmp(two, one, shallow=False)
    out["count_rows"] = sum(1 for _ in open(one))
    out["one_pass_pairs_per_s"] = args.reads / min(out["one_pass_s"])
    print(json.dumps(out))
    if not out["counts_identical"] or any(out["rc"]):
        sys.exit(4)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reads", type=int, default=2_000_000)
    ap.add_argument("--out-dir", default="/tmp/nb200_file_bench")
    ap.add_argument("--gpus", type=int, default=1, help="GPUs of the node for `align` (one process, nb200_align_files_multi)")
    ap.add_argument("--cores", type=int, default=0, help="host threads (0 = all)")
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg4"], help="cfg4: combined MHC + KIR + transcript library, 80 k cells")
    ap.add_argument("--compare-1gpu", action="store_true", help="also run on ONE GPU and require a byte-identical per-read TSV")
    ap.add_argument("--skip-report", action="store_true")
    ap.add_argument("--rss", action="store_true", help="run the `aligner` executable as a child process on the same input and report its peak RSS "
                                                       "(the streaming pipeline holds a fixed pool of slabs, not the file)")
    ap.add_argument("--counts", action="store_true", help="time the two-step route (align + report) against the fused `align --counts`, "
                                                          "alternating, two repetitions each, and compare the counts files")
    ap.add_argument("--tenx", action="store_true", help="raw 10x R1 / R2 FASTQ (plain gzip) + whitelist: fastq-to-bam then align --counts "
                                                        "on its BAM against fastq-to-counts, alternating; wall clock, peak RSS, identical counts")
    args = ap.parse_args()
    os.makedirs(args.out_dir, exist_ok=True)
    if args.workload == "cfg4":
        lib, codes = synth.combined_library(n_transcripts=3000, seed=4)
        n_cells = 80000
    else:
        lib, codes = synth.allele_family_library(n_founders=40, alleles_per_founder=50, length=1098, snps_mean=15.0, seed=1)
        n_cells = 10000
    lib_path = os.path.join(args.out_dir, "lib.json")
    with open(lib_path, "w") as f:
        json.dump(lib, f)
    if args.tenx:
        tenx_bench(args, lib_path)
        return
    bam = os.path.join(args.out_dir, "in.bam")
    made = {"workload": args.workload, "reads": args.reads}
    try:                                    # the same input as an earlier run into this directory: not written again
        reuse = json.load(open(bam + ".json")) == made and os.path.exists(bam)
    except (OSError, ValueError):
        reuse = False
    t0 = time.time()
    if reuse:
        nbytes = os.path.getsize(bam)
    else:
        nbytes = write_bam_chunked(bam, codes, args.reads, n_cells)
        with open(bam + ".json", "w") as f:
            json.dump(made, f)
    print("%s %s: %d reads, %.0f MB in %.1fs" % ("reused" if reuse else "wrote", bam, args.reads, nbytes / 1e6, time.time() - t0), file=sys.stderr)
    from nimble_b200.engine import Engine
    eng = Engine(0, args.cores)
    tsv = os.path.join(args.out_dir, "out.tsv")
    kw = {"engine": eng} if args.gpus <= 1 else {"gpus": args.gpus}
    if args.counts:
        counts_bench(args, eng, kw, lib_path, bam, tsv, nbytes)
        return
    frontend.align(lib_path, tsv, [bam], args.cores, "unstranded", "", None, **kw)          # warm-up (CUDA context, page cache)
    os.remove(tsv)                          # the timed run writes a fresh file (replacing a GB-sized one costs 0.2-0.4 s of unlink alone)
    t0 = time.perf_counter()
    rc = frontend.align(lib_path, tsv, [bam], args.cores, "unstranded", "", None, **kw)
    t_align = time.perf_counter() - t0
    out = {"workload": args.workload, "reads": args.reads, "rc": rc, "align_s": t_align, "align_reads_per_s": args.reads / t_align,
           "bam_mb": nbytes / 1e6, "tsv_mb": os.path.getsize(tsv) / 1e6, "host_threads": args.cores or os.cpu_count(), "gpus": args.gpus}
    if args.compare_1gpu and args.gpus > 1:
        tsv1 = os.path.join(args.out_dir, "out_1gpu.tsv")
        t0 = time.perf_counter()
        frontend.align(lib_path, tsv1, [bam], args.cores, "unstranded", "", None, engine=eng)
        out["align_s_1gpu"] = time.perf_counter() - t0
        out["align_reads_per_s_1gpu"] = args.reads / out["align_s_1gpu"]
        import filecmp
        out["tsv_identical_to_1gpu"] = filecmp.cmp(tsv, tsv1, shallow=False)
        os.remove(tsv1)
    if args.rss:
        import resource
        import subprocess
        exe = os.path.join(ROOT, "nimble_b200", "aligner")
        before = resource.getrusage(resource.RUSAGE_CHILDREN).ru_maxrss
        t0 = time.perf_counter()
        rc2 = subprocess.call([exe, "--input", bam, "-c", str(args.cores or os.cpu_count()), "--strand_filter", "unstranded", "-r", lib_path,
                               "-o", os.path.join(args.out_dir, "out_child.tsv")] + (["--gpus", str(args.gpus)] if args.gpus > 1 else []))
        out["aligner_process_s"] = time.perf_counter() - t0           # includes CUDA context creation and the index build
        out["aligner_rc"] = rc2
        out["aligner_peak_rss_mb"] = max(before, resource.getrusage(resource.RUSAGE_CHILDREN).ru_maxrss) / 1024.0
        os.remove(os.path.join(args.out_dir, "out_child.tsv"))
    if not args.skip_report:
        t0 = time.perf_counter()
        frontend.report(tsv, os.path.join(args.out_dir, "counts.tsv"), None, 0.05, False, engine=eng)
        out["report_s"] = time.perf_counter() - t0
        out["count_rows"] = sum(1 for _ in open(os.path.join(args.out_dir, "counts.tsv")))
    print(json.dumps(out))
    if out.get("tsv_identical_to_1gpu") is False:
        sys.exit(4)


if __name__ == "__main__":
    main()
