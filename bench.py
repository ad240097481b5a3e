#!/usr/bin/env python
"""Headline benchmark: reads/sec of nimble's read-assignment hot path on B200.

Workload (BASELINE.json configs[1]): synthetic 10x 3' scRNA-seq, 10 M reads x 90 bp with CB/UB
keys vs a synthetic MHC-I allele-family library (40 genes x 50 alleles, 1098 bp), default
library config.  A step = one pass of the whole path over the batch: k-mer probe +
equivalence-class intersection -> banded Smith-Waterman -> score/feature filter -> per-cell UMI
aggregation -> count table.  Weak scaling: every rank owns 10 M reads of its own cell shard.

  python bench.py [--gpus N --steps K --warmup W]            # CUDA path (one JSON line)
  python bench.py --impl reference [...]                      # CPU arm (oracle, all host threads)
  python bench.py --dump-outputs DIR [...]                    # also writes the last timed step's count table (.npy)
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from nimble_b200 import shard, synth  # noqa: E402

WORKLOAD = "cfg2: synthetic 10x 3' scRNA-seq, 90bp reads + CB/UB vs MHC-like allele-family library (40x50 alleles, 1098bp), default config"
METRIC = "reads/sec (device-timed, 1/2/4/8 B200) vs MHC-like lib; SW GCUPS; HBM GB/s"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# The driver reads exactly ONE JSON line from stdout.  Libraries (NCCL prints its version banner on
# stdout) must not leak into it: fd 1 is pointed at stderr for the whole run and the JSON line goes to
# the saved descriptor.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(line):
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.idx = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for nm, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "power_w_max": max(pw) if pw else None, "samples": len(sm)}


WORKLOAD5 = "cfg5: synthetic transcriptome library (%d transcripts, ~2 kb, 30%% sharing exon blocks), k=31, score_percent 0.25, 100bp reads + CB/UB"


WORKLOAD4 = ("cfg4 (scaled per GPU): synthetic scRNA-seq 90bp reads + CB/UB, sharded by cell barcode, vs ONE combined library "
             "(2000 MHC-like + 1530 KIR-like alleles + 3000 immune-gene transcripts), union feature-calling")
WORKLOAD3 = ("cfg3 (scaled): synthetic bulk paired-end 2x150bp vs KIR-like library (17 genes x 90 alleles, 1350bp), "
             "num_mismatches 0, --strand_filter fiveprime, intersect_level 2, no cell barcodes (counts per feature set)")


def make_workload(n_reads, rank, world, n_cells=10000, kind="cfg2", transcripts=50000):
    """Returns (library json, r1 ascii, r2 ascii or None, key or None)."""
    t0 = time.time()
    if kind == "cfg3":
        lib, codes = synth.allele_family_library(n_founders=17, alleles_per_founder=90, length=1350, snps_mean=12.0, seed=3,
                                                 name_prefix="KIR", config={"num_mismatches": 0, "intersect_level": 2})
        a1, a2, _ = synth.sample_pairs(codes, n_reads, read_len=150, insert_mean=300, insert_sd=50, err_rate=0.005,
                                       off_target=0.1, seed=3 + 1000 * rank)
        log("[rank %d] workload cfg3: %d pairs generated in %.1fs" % (rank, n_reads, time.time() - t0))
        return lib, a1, a2, None
    if kind == "cfg4":
        # MHC-like + KIR-like + immune-gene transcripts in ONE library (6.5 k sequences), union feature-calling
        lib, codes = synth.combined_library(n_transcripts=3000, seed=4)
        asc, truth = synth.sample_reads(codes, n_reads, read_len=90, err_rate=0.005, off_target=0.2, rc_frac=0.1,
                                        seed=4 + 1000 * rank)
        n_cells = 80000 // max(1, world) if world > 1 else 10000
    if kind == "cfg5":
        lib, codes = synth.random_transcript_library(n_seqs=transcripts, mean_len=2000, family_frac=0.3, seed=5,
                                                     config={"score_percent": 0.25})
        asc, truth = synth.sample_reads(codes, n_reads, read_len=100, err_rate=0.005, off_target=0.2, rc_frac=0.1,
                                        seed=6 + 1000 * rank)
    elif kind != "cfg4":
        lib, codes = synth.allele_family_library(n_founders=40, alleles_per_founder=50, length=1098, snps_mean=15.0, seed=1)
        asc, truth = synth.sample_reads(codes, n_reads, read_len=90, err_rate=0.005, off_target=0.2, rc_frac=0.1,
                                        seed=2 + 1000 * rank)
    # cells of this rank's shard: draw candidates, keep those hashing to `rank`
    rng = np.random.default_rng(77 + rank)
    pool = np.zeros(0, np.uint64)
    while len(pool) < n_cells:
        cand = rng.integers(0, 1 << 32, size=n_cells * max(2, world) * 2, dtype=np.uint64)
        keep = shard.shard_of_key(cand << np.uint64(32), world) == rank
        pool = np.concatenate([pool, cand[keep]])
    pool = pool[:n_cells]
    key = synth.barcodes_10x(n_reads, n_cells=n_cells, seed=2 + 1000 * rank, truth=truth)
    # remap the generator's random cells onto this rank's pool (same cell -> same pool entry)
    cells, inv = np.unique(key >> np.uint64(32), return_inverse=True)
    key = (pool[np.arange(len(cells)) % len(pool)][inv] << np.uint64(32)) | (key & np.uint64(0xFFFFFFFF))
    log("[rank %d] workload %s: %d reads generated in %.1fs" % (rank, kind, n_reads, time.time() - t0))
    return lib, asc, None, key


DUMP_BYTES = 64_000_000         # all files of one --dump-outputs, .npy headers included


def dump_outputs(out_dir, table, limit=DUMP_BYTES, prefix=""):
    """Writes the count table of the last timed step, as a caller of the timed path receives it, to out_dir/<name>.npy
    in float64 (exact for its uint32 values): cell, count, feat_off, feat_ids and the 0-d dropped_empty, n_called,
    n_umis.  A table larger than `limit` bytes is written as a sample of its rows drawn with a fixed seed from the row
    count alone: rows.npy holds the sampled row indices (ascending), feat_off / feat_ids describe those rows only."""
    n = len(table.cell)
    off = table.feat_off.astype(np.int64)
    out = {"cell": table.cell, "count": table.count, "feat_off": off, "feat_ids": table.feat_ids}
    nbytes = lambda d: sum(128 + 8 * v.size for v in d.values()) + 3 * (128 + 8)      # 128 B header per .npy file
    m = n
    while nbytes(out) > limit:
        m = int(m * 0.95 * limit / nbytes(out))
        rows = np.sort(np.random.default_rng(0).choice(n, size=m, replace=False))
        nf = off[rows + 1] - off[rows]
        ends = np.cumsum(nf)
        ids = np.repeat(off[rows] - (ends - nf), nf) + np.arange(int(ends[-1]) if m else 0)
        out = {"rows": rows, "cell": table.cell[rows], "count": table.count[rows],
               "feat_off": np.concatenate([[0], ends]), "feat_ids": table.feat_ids[ids]}
    for k_ in ("dropped_empty", "n_called", "n_umis"):
        out[k_] = np.array(getattr(table, k_))
    os.makedirs(out_dir, exist_ok=True)
    for k_, v in out.items():
        np.save(os.path.join(out_dir, prefix + k_ + ".npy"), np.asarray(v, np.float64))
    log("[dump] %d of %d count rows -> %s" % (m, n, out_dir))


def host_threads():
    """All host threads this process may use (torchrun exports OMP_NUM_THREADS=1: ignore that)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def pin_to_gpu_numa_node(gpu_index):
    """One process per GPU: run on the cores next to that GPU (NVML's ideal CPU affinity) so that the pinned
    host buffers are first-touched on its NUMA node and the count-table D2H does not cross sockets."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, v in enumerate(words) for b in range(64) if (v >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            log("[gpu %d] pinned to %d cores (%d..%d)" % (gpu_index, len(cpus), min(cpus), max(cpus)))
    except Exception as e:      # best effort
        log("[gpu %d] no CPU affinity set: %s" % (gpu_index, e))


def oracle_pass(O, lo, asc, key, threads, asc2=None):
    """One CPU pass of the same path (oracle): align + UMI aggregation.  Returns seconds."""
    n = asc.shape[0]
    off = np.arange(0, asc.size + 1, asc.shape[1], dtype=np.int64)
    t0 = time.perf_counter()
    r2 = None if asc2 is None else (asc2.reshape(-1), off)
    res, feats = O.align(lo, (asc.reshape(-1), off), r2, n_threads=threads)
    if key is None:
        key = np.zeros(n, np.uint64)
    nf = res["n_feat"].astype(np.int64)
    foff = np.zeros(n + 1, np.int32)
    np.cumsum(nf, out=foff[1:])
    ids = feats[np.arange(feats.shape[1])[None, :] < nf[:, None]].astype(np.uint32)
    t1 = time.perf_counter()
    O.a6_ids(key, foff, ids, None, lo.tok_end, lo.tok_comma, 0.05, False, n_threads=threads)
    t2 = time.perf_counter()
    oracle_pass.last = {"align_s": t1 - t0, "a6_s": t2 - t1}
    return t2 - t0


def parity_slice(eng, lg, lib_json, asc, asc2, key, kmer, strand, threads, n=100_000):
    """Before anything is timed: the first `n` reads of THIS workload through the CUDA path (C ABI) and through the
    oracle; per-read records, feature calls and the count table must agree bit for bit.  Aborts the run otherwise."""
    from oracle import oracle as O
    O.build()
    n = min(n, asc.shape[0])
    a1 = asc[:n]
    a2 = None if asc2 is None else asc2[:n]
    kk = None if key is None else np.ascontiguousarray(key[:n])
    off = np.arange(0, a1.size + 1, a1.shape[1], dtype=np.int64)
    t0 = time.perf_counter()
    lo = O.Library(lib_json, k=kmer, strand_filter=strand)
    ro, fo = O.align(lo, (a1.reshape(-1), off), None if a2 is None else (a2.reshape(-1), off), n_threads=threads)
    table, rg, fg = eng.align(lg, a1, a2, key=kk, per_read=True)
    bad = [f for f in ro.dtype.names if not np.array_equal(ro[f], rg[f])]
    if not np.array_equal(fo, fg):
        bad.append("feature ids")
    nf = ro["n_feat"].astype(np.int64)
    foff = np.zeros(n + 1, np.int32)
    np.cumsum(nf, out=foff[1:])
    ids = fo[np.arange(fo.shape[1])[None, :] < nf[:, None]].astype(np.uint32)
    if kk is not None:
        cell, cnt, o_off, o_ids, dropped = O.a6_ids(kk, foff, ids, None, lo.tok_end, lo.tok_comma, 0.05, False, n_threads=threads)
        if not (np.array_equal(cell, table.cell) and np.array_equal(cnt, table.count) and np.array_equal(o_ids, table.feat_ids)
                and np.array_equal(o_off.astype(np.int64), table.feat_off.astype(np.int64)) and dropped == table.dropped_empty):
            bad.append("count table")
    else:               # bulk data: one count per distinct feature set
        hist = {}
        for i in np.nonzero(nf)[0]:
            t = tuple(int(x) for x in fo[i, :nf[i]])
            hist[t] = hist.get(t, 0) + 1
        got = {tuple(int(x) for x in table.feat_ids[table.feat_off[i]:table.feat_off[i + 1]]): int(table.count[i])
               for i in range(len(table))}
        if got != hist:
            bad.append("count table")
    out = {"reads": int(n), "ok": not bad, "called": int((ro["reason"] == 0).sum()), "sw_orientations": int(ro["n_sw"].sum()),
           "count_rows": int(len(table)), "seconds": round(time.perf_counter() - t0, 2),
           "checked": "every nb200_read_result field + feature ids per read + count table vs oracle/nimble_oracle.c"}
    if bad:
        out["mismatch"] = bad
        log("PARITY SLICE FAILED: %s" % bad)
        emit({"metric": METRIC, "parity_slice": out, "error": "CUDA path differs from the oracle; nothing was timed"})
        raise SystemExit(3)
    return out


def run_reference(args, rank, world):
    """CPU arm: the oracle port of the reference path (the real aligner is not installable offline,
    BASELINE.md §2) on all host threads, bounded sample per step."""
    if rank != 0:
        return
    from oracle import oracle as O
    O.build()
    sample = int(args.ref_sample)
    lib, asc, _, key = make_workload(sample, 0, 1)
    lo = O.Library(lib, k=20)
    ix = lo.index
    threads = host_threads()
    for _ in range(args.warmup):
        oracle_pass(O, lo, asc, key, threads)
    t = 0.0
    for _ in range(args.steps):
        t += oracle_pass(O, lo, asc, key, threads)
    ms = 1e3 * t / max(1, args.steps)
    val = sample / (ms / 1e3)
    st = getattr(oracle_pass, "last", {"align_s": 0.0, "a6_s": 0.0})
    index = {"n_refs": len(lo.names), "n_kmers": ix.n_kmers, "n_classes": ix.n_classes}
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "reads/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u64/s16", "data": "synthetic",
            "config": make_config(WORKLOAD, "cfg2", args.reads, asc.shape[1], 20, index, max(1, args.gpus), False),
            "cpu_baseline": {"value": val, "unit": "reads/s", "cores": threads, "kind": "port",
                             "sample": "%d reads of the cfg2 workload per step (oracle/nimble_oracle.c): orc_align on %d OpenMP threads "
                                       "(%.0f ms of the last step), orc_a6_mt on %d threads (cells dealt to threads, %.0f ms)"
                                       % (sample, threads, 1e3 * st["align_s"], threads, 1e3 * st["a6_s"])},
            "e2e": {"value": val, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def run_barcodes(args, rank, world, local):
    """Secondary line (SURVEY.md §8f rank 2): `nimble fastq-to-bam`'s cell-barcode correction.
    A step = correct_cell_barcode over one batch of raw 16-mers + qualities against the whitelist."""
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — nimble_b200 has no CPU path")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import nimble_b200
    eng = nimble_b200.Engine(local)
    n, n_wl = args.reads, args.whitelist
    t0 = time.time()
    wl_a, cb, q = synth.barcode_workload(n, n_whitelist=n_wl, seed=11 + 1000 * rank)
    wl_s = [bytes(r).decode() for r in wl_a]
    log("[rank %d] barcode workload: %d reads, %d whitelist entries in %.1fs" % (rank, n, n_wl, time.time() - t0))
    wl = eng.load_whitelist(wl_s, 16)
    cbp = eng.pinned_empty(cb.size).reshape(cb.shape); cbp[:] = cb
    qp = eng.pinned_empty(q.size).reshape(q.shape); qp[:] = q
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import oracle as O
        O.build()
        ns = min(n, args.cpu_sample)
        t0 = time.perf_counter()
        O.cb_correct(wl_s, cb[:ns], q[:ns], None, 16)
        sec = time.perf_counter() - t0
        cpu_baseline = {"value": ns / sec, "unit": "reads/s", "cores": 1, "kind": "port",
                        "sample": "first %d reads, oracle/cb_oracle.c (sequential like the reference's cache loop), %.1fs incl. whitelist set build" % (ns, sec)}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    eng.cb_upload(wl, cbp, qp)
    sampler = ClockSampler(local)
    sampler.start()                       # steps are ~1 ms: give nvidia-smi the warm-up to start sampling
    for _ in range(max(args.warmup, 50)):
        eng.correct_barcodes_resident(wl, fetch=False)
    barrier()
    ms, acc = 0.0, {}
    for _ in range(args.steps):
        _, _, st = eng.correct_barcodes_resident(wl, fetch=False)
        ms += st["kernel_ms"]
        for k_, v in st.items():
            acc[k_] = acc.get(k_, 0) + v
    barrier()
    clocks = sampler.stop()
    outp = (eng.pinned_empty(4 * n, np.int32), eng.pinned_empty(n, np.uint8))
    for _ in range(2):
        eng.correct_barcodes(wl, cbp, qp, out=outp)
    barrier()
    w0 = time.perf_counter()
    for _ in range(args.steps):
        idx, status, st_e = eng.correct_barcodes(wl, cbp, qp, out=outp)
    barrier()
    e2e_ms = 1e3 * (time.perf_counter() - w0) / args.steps
    stats = torch.tensor([ms / args.steps, e2e_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
    ms_step, e2e_ms = (float(x) for x in stats.tolist())
    if rank == 0:
        peak, peak_src = peaks()
        K = args.steps
        # algorithmic bytes per read of the whole pipeline: 16 B barcode in, 8 B key + 4 B index + 1 B status out,
        # one 32 B whitelist sector per probe (device-counted), 16 B qualities for the reads that missed
        alg = n * (16 + 8 + 4 + 1) + acc["probes"] / K * 32 + acc["n_exact_miss"] / K * 16
        line = {"metric": "reads/sec (fastq-to-bam cell-barcode correction)", "value": world * n / (ms_step / 1e3), "unit": "reads/s",
                "n_gpus": world, "steps": K, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "u64 3-bit packed barcodes / u8 qualities", "data": "synthetic",
                "config": {"workload": "fastq-to-bam: %d raw 16-mer barcodes + qualities vs %d-entry whitelist (10x-like errors)" % (n, n_wl),
                           "table_mb": wl.table_bytes / 1e6, "l2": "inputs larger than L2 (%.0f MB per pass)" % (n * 32 / 1e6),
                           "stats": "includes the distinct-raw-barcode count (radix sort) the reference prints"},
                "clocks": clocks,
                "e2e": {"value": world * n / (e2e_ms / 1e3), "unit": "reads/s", "h2d_bytes_per_step": int(st_e["h2d_bytes"]),
                        "d2h_bytes_per_step": int(st_e["d2h_bytes"]), "ms_per_step": e2e_ms,
                        "api": "nb200_correct_barcodes (C ABI, pinned host buffers in, index + status out)"},
                "gpu_launches": int(acc["launches"]),
                "roofline": {"kernel": "cb_exact_kernel + cb_hamming_kernel + distinct count (whole pipeline)", "bound": "hbm",
                             "achieved": alg / (ms_step / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                             "frac": alg / (ms_step / 1e3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                             "algorithmic_bytes_per_step": alg},
                "cpu_baseline": cpu_baseline,
                "barcodes": {k_: acc[k_] / K for k_ in ("cb_perfect_match", "cb_corrected", "cb_no_correction", "n_exact_miss",
                                                        "n_multi", "probes", "cache_size")}}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def run_report(args, rank, world, local):
    """Secondary line (SURVEY.md §8a A6): `nimble report`'s UMI stage alone.  A step = per-read rows
    (cell, umi, feature list) of the headline workload -> per-cell counts (merge, per-UMI thresholding,
    intersection, count): nb200_umi_counts."""
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — nimble_b200 has no CPU path")
    torch.cuda.set_device(local)
    import nimble_b200
    eng = nimble_b200.Engine(local)
    lib_json, asc, _, key = make_workload(args.reads, rank, world)
    lg = eng.load_library(lib_json, k=20)
    table0, res, feats = eng.align(lg, asc, key=key, per_read=True)
    called = np.nonzero(res["n_feat"])[0]
    nf = res["n_feat"][called].astype(np.int64)
    off = np.zeros(len(called) + 1, np.uint32)
    np.cumsum(nf, out=off[1:])
    ids = feats[called][np.arange(feats.shape[1])[None, :] < nf[:, None]].astype(np.uint32)
    rkey = np.ascontiguousarray(key[called])
    m = len(called)
    log("[rank %d] report workload: %d per-read rows with a call (of %d reads), %d feature ids" % (rank, m, len(asc), len(ids)))
    cpu_baseline = None
    if rank == 0 and not args.no_cpu_baseline:
        from oracle import oracle as O
        O.build()
        lo = O.Library(lib_json, k=20)
        ns = min(m, args.cpu_sample)
        t0 = time.perf_counter()
        O.a6_ids(rkey[:ns], off[:ns + 1].astype(np.int32), ids[:off[ns]], None, lo.tok_end, lo.tok_comma, 0.05, False)
        sec = time.perf_counter() - t0
        cpu_baseline = {"value": ns / sec, "unit": "rows/s", "cores": 1, "kind": "port",
                        "sample": "first %d rows, oracle/nimble_oracle.c orc_a6 (sort + per-UMI loop), %.1fs; the reference's pandas "
                                  "report() iterates UMI groups in Python (O(10^3) groups/s)" % (ns, sec)}
    for _ in range(args.warmup):
        eng.umi_counts(lg, rkey, off, ids)
    sampler = ClockSampler(local)
    sampler.start()
    torch.cuda.synchronize()
    ms, launches, w0 = 0.0, 0, time.perf_counter()
    for _ in range(args.steps):
        table = eng.umi_counts(lg, rkey, off, ids)
        t = eng.timing()
        ms += t["agg_ms"]; launches += t["launches"]
    wall_ms = 1e3 * (time.perf_counter() - w0) / args.steps
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, table)
    ms /= args.steps
    same = np.array_equal(table.cell, table0.cell) and np.array_equal(table.count, table0.count) and np.array_equal(table.feat_ids, table0.feat_ids)
    peak, peak_src = peaks()
    width = lg.config.max_hits_to_report
    # streamed bytes of the stage (rows m, groups ~m/3): padded feature rows in, the sort passes (key+value per pass), table out
    alg = m * (4 * width + 2 + 8) + 2 * m * 8 * (2 * ((width + 1) // 2) + 8) + t["d2h_bytes"]
    emit({"metric": "rows/sec (report: per-UMI thresholding + intersection + per-cell counts)", "value": m / (ms / 1e3), "unit": "rows/s",
          "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
          "vs_baseline": None, "dtype": "u32 ids / u64 keys / f64 thresholds (Kahan)", "data": "synthetic",
          "config": {"workload": "report: the %d called rows of the cfg2 workload (%d reads), 10 000 cells" % (m, len(asc)),
                     "l2": "inputs larger than L2 (%.0f MB of rows per pass)" % (m * (4 * width + 10) / 1e6)},
          "clocks": clocks,
          "e2e": {"value": m / (wall_ms / 1e3), "unit": "rows/s", "h2d_bytes_per_step": int(t["h2d_bytes"]),
                  "d2h_bytes_per_step": int(t["d2h_bytes"]), "ms_per_step": wall_ms,
                  "api": "nb200_umi_counts (C ABI, host rows in, count table out)"},
          "gpu_launches": int(launches),
          "roofline": {"kernel": "A6 pipeline (radix sorts + umi_kernel + run-length count)", "bound": "hbm", "achieved": alg / (ms / 1e3) / 1e9,
                       "peak": peak, "unit": "GB/s", "frac": alg / (ms / 1e3) / 1e9 / peak, "traffic": None, "peak_source": peak_src},
          "cpu_baseline": cpu_baseline, "count_rows": len(table), "equals_align_table": bool(same)})


def pack_stride(read_len):
    words = max(1, (read_len + 31) // 32)
    return (12 * words + 15) & ~15


def make_config(workload_name, kind, n_reads, read_len, kmer, index, world, paired):
    """`config` of the JSON line.  Both arms print the same dict (the reference arm runs a bounded sample of this
    workload and says so in cpu_baseline.sample)."""
    return {"workload": workload_name, "reads_per_gpu": int(n_reads), "read_len": int(read_len), "k": int(kmer),
            "n_refs": int(index["n_refs"]), "n_kmers": int(index["n_kmers"]), "n_classes": int(index["n_classes"]),
            "parallelism": "cell-barcode shard x%d, index replicated" % world,
            "l2": "inputs larger than L2 (%.0f MB packed reads per pass)"
                  % (n_reads * pack_stride(read_len) * (2 if paired else 1) / 1e6)}


def ncu_traffic(kernel_prefix, workload):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of a kernel, from the committed summary
    scripts/ncu_summary.py writes out of an `ncu --set full` report (profiles/r02_ncu_summary.json)."""
    p = os.path.join(ROOT, "profiles", "r02_ncu_summary.json")
    try:
        with open(p) as f:
            d = json.load(f)
        if d.get("workload") != workload:
            return None, None
        for k_ in d.get("kernels", []):
            if k_["name"].startswith(kernel_prefix):
                return float(k_["dram_bytes"]), {"reads_per_launch": d.get("reads_per_launch"), "source": "profiles/r02_ncu_summary.json",
                                                 "issue_active_pct": k_.get("issue_active_pct"),
                                                 "warp_inst_per_read": k_.get("warp_inst_per_read"),
                                                 "threads_per_inst": k_.get("threads_per_inst")}
    except Exception:
        pass
    return None, None


def probe_roofline(eng, info, avg, n, packed, packed2, width, peak, peak_src, workload_kind, ra_hbm=None):
    """Roofline block of probe_kernel.  SURVEY.md §8(d): algorithmic bytes per read = P x 16 B (one table entry per lookup,
    P device-counted) + packed read in (stride bytes) + 8 B key + 16 B result; the 32 B-sector variant is reported beside it."""
    mates = 2 if packed2 is not None else 1
    per_launch = (1 << 20) if packed2 is not None else (1 << 21)      # reads per probe_kernel launch (engine batch)
    # the roofline's kernel is probe_kernel itself (CUDA events around its launches); probe_ms is the whole probe stage
    # (probe_kernel + the calling kernels that run behind it on the same stream)
    stage_s = avg["probe_ms"] / 1e3
    probe_s = (avg.get("probe_kernel_ms") or avg["probe_ms"]) / 1e3
    io_bytes = n * (packed.device_stride * mates + 8 + 16)      # the kernel reads full records (compact ones are expanded on arrival)
    alg = avg["probes"] * 16 + io_bytes
    alg32 = avg["probes"] * 32 + io_bytes
    ach = alg / probe_s / 1e9 if probe_s > 0 else 0.0
    ra_table = eng.random_access_bandwidth(max(info["table_bytes"], 1 << 24))
    if ra_hbm is None:
        ra_hbm = eng.random_access_bandwidth(8 << 30)
    resident = "L2-resident" if info["table_bytes"] < 100e6 else "HBM-resident"
    useful_gbs = avg["probes"] * 32 / probe_s / 1e9 if probe_s > 0 else 0.0            # one 32 B sector per LOOKUP (useful)
    sector_gbs = avg["probe_slots"] * 32 / probe_s / 1e9 if probe_s > 0 else 0.0       # sectors actually read (incl. second buckets)
    traffic, ncu = ncu_traffic("probe_kernel", workload_kind)
    scale = min(n, per_launch) / max(n, 1)
    out = {"kernel": "probe_kernel (k-mer extract + canonical hash probe + eq-class AND + feature call)", "bound": "hbm",
           "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
           "traffic": traffic * min(n, per_launch) / ncu["reads_per_launch"] if traffic and ncu and ncu.get("reads_per_launch") else None,
           "algorithmic_bytes_per_launch": alg * scale, "algorithmic_bytes_per_read": alg / max(n, 1),
           "launches_per_step": (n + per_launch - 1) // per_launch, "ms_per_step": probe_s * 1e3,
           "stage": {"what": "probe stage = probe_kernel + call_fast + sw_setup + call_slow + wide kernels (same stream, back to back)",
                     "ms_per_step": avg["probe_ms"], "achieved": alg / stage_s / 1e9 if stage_s > 0 else 0.0,
                     "frac": alg / stage_s / 1e9 / peak if stage_s > 0 else 0.0},
           "peak_source": peak_src,
           "sector_variant": {"achieved": alg32 / probe_s / 1e9 if probe_s > 0 else 0.0, "frac": alg32 / probe_s / 1e9 / peak if probe_s > 0 else 0.0,
                              "what": "same formula with 32 B (one L2 sector) per lookup instead of the 16 B entry"},
           "limited_by": ("instruction issue: the %.0f MB table is L2-resident, DRAM traffic is a fraction of the algorithmic bytes"
                          % (info["table_bytes"] / 1e6)) if resident == "L2-resident" else "HBM random access (32 B sectors)",
           "ncu": ncu,
           "random_access": {"what": "independent random 32 B-sector gathers, measured in this run (nb200_bench_random_access)",
                             "table_sized_gbs": ra_table[0], "hbm_8gib_gbs": ra_hbm[0],
                             "useful_gbs": useful_gbs, "sectors_read_gbs": sector_gbs,
                             "sectors_per_lookup": avg["probe_slots"] / max(1.0, avg["probes"]),
                             "frac_of_table_sized": useful_gbs / ra_table[0] if ra_table[0] else None,
                             "frac_of_hbm_random": useful_gbs / ra_hbm[0] if ra_hbm[0] else None,
                             "note": "useful = one sector per lookup; sectors a lookup reads beyond its first are not counted as achieved"},
           "note": "table is %.0f MB (%s)" % (info["table_bytes"] / 1e6, resident)}
    return out, ra_hbm


def hbm_pass(eng, args, threads, peak, peak_src, ra_hbm):
    """Short HBM-resident pass appended to the default run: cfg5-shaped library (transcript families, k = 31,
    score_percent 0.25) whose table is far larger than L2, so that the probe's fraction of the measured HBM
    random-access rate lands in the same record.  Parity slice first, like every timed workload."""
    T = args.hbm_transcripts
    t0 = time.time()
    lib, codes = synth.random_transcript_library(n_seqs=T, mean_len=2000, family_frac=0.3, seed=5, config={"score_percent": 0.25})
    n = args.hbm_reads
    asc, truth = synth.sample_reads(codes, n, read_len=100, err_rate=0.005, off_target=0.2, rc_frac=0.1, seed=6)
    key = synth.barcodes_10x(n, n_cells=10000, seed=6, truth=truth)
    lg = eng.load_library(lib, k=31)
    info = lg.info
    log("[hbm pass] %d transcripts: %s, built in %.1fs" % (T, info, time.time() - t0))
    par = parity_slice(eng, lg, lib, asc, None, key, 31, "unstranded", threads, n=args.hbm_parity) if not args.no_cpu_baseline else None
    packed = eng.pack(asc, pinned=True)
    kp = eng.pinned_empty(8 * n, np.uint64)
    kp[:] = key
    eng.upload(packed, None, key=kp)
    for _ in range(2):
        eng.align_resident(lg, fetch_counts=False)
    eng.set_overlap(False)
    acc, K = {}, args.steps
    for _ in range(K):
        eng.align_resident(lg, fetch_counts=False)
        for k_, v in eng.timing().items():
            acc[k_] = acc.get(k_, 0) + v / K
    eng.set_stats(True)                  # lookups / sectors: one more pass with the device counters on
    eng.align_resident(lg, fetch_counts=False)
    ts = eng.timing()
    acc["probes"], acc["probe_slots"] = ts["probes"], ts["probe_slots"]
    eng.set_overlap(True)
    eng.set_stats(False)
    roof, _ = probe_roofline(eng, info, acc, n, packed, None, lg.config.max_hits_to_report, peak, peak_src, "cfg5", ra_hbm)
    roof["workload"] = WORKLOAD5 % T
    roof["reads"] = n
    roof["steps"] = K
    roof["reads_per_s_resident"] = n / (acc["total_ms"] / 1e3)
    roof["kernels_ms"] = {k_: acc[k_ + "_ms"] for k_ in ("probe", "probe_kernel", "sw", "call", "agg", "total")}
    roof["parity_slice"] = par
    return roof


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--reads", type=int, default=int(os.environ.get("NB200_BENCH_READS", 10_000_000)))
    ap.add_argument("--ref-sample", type=int, default=int(os.environ.get("NB200_REF_SAMPLE", 2_000_000)))
    ap.add_argument("--cpu-sample", type=int, default=int(os.environ.get("NB200_CPU_SAMPLE", 2_000_000)))
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the oracle legs (cpu_baseline AND parity slices): profiling runs only")
    ap.add_argument("--whitelist", type=int, default=737_280, help="fastq-to-bam: whitelist entries (737280 = 10x v2, 6794880 = v3)")
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg3", "cfg4", "cfg5", "fastq-to-bam", "report"],
                    help="cfg2 = BASELINE.json configs[1] (default, the headline); cfg5 = HBM-resident transcriptome-scale table")
    ap.add_argument("--transcripts", type=int, default=50000, help="cfg5: number of synthetic transcripts")
    ap.add_argument("--parity-reads", type=int, default=100_000, help="reads of the workload diffed against the oracle before timing")
    ap.add_argument("--hbm-transcripts", type=int, default=int(os.environ.get("NB200_BENCH_HBM_TRANSCRIPTS", 25000)),
                    help="default run: transcripts of the appended HBM-resident pass (0 = skip)")
    ap.add_argument("--hbm-reads", type=int, default=4_000_000)
    ap.add_argument("--hbm-parity", type=int, default=20_000)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the count table of the last one to DIR/<name>.npy (float64, at most 64 MB: "
                         "a seeded sample of the rows beyond that) to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload == "fastq-to-bam"):
        ap.error("--dump-outputs: the timed path of --impl reference and --workload fastq-to-bam returns no count table")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    args.warmup = max(3, args.warmup)
    if args.workload == "fastq-to-bam":
        run_barcodes(args, rank, world, local)
        return
    if args.workload == "report":
        run_report(args, rank, world, local)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — nimble_b200 has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        pin_to_gpu_numa_node(local)

    import nimble_b200
    eng = nimble_b200.Engine(local)
    kmer = 31 if args.workload == "cfg5" else 20
    lib_json, asc, asc2, key = make_workload(args.reads, rank, world, kind=args.workload, transcripts=args.transcripts)
    workload = {"cfg2": WORKLOAD, "cfg3": WORKLOAD3, "cfg4": WORKLOAD4}.get(args.workload) or WORKLOAD5 % args.transcripts
    strand = "fiveprime" if args.workload == "cfg3" else "unstranded"
    n = asc.shape[0]
    read_len = asc.shape[1]
    t0 = time.time()
    lg = eng.load_library(lib_json, strand_filter=strand, k=kmer)
    info = lg.info
    log("[rank %d] library: %s built+uploaded in %.1fs" % (rank, info, time.time() - t0))
    threads = max(1, host_threads() // (world if world > 1 else 1))

    # ---- parity first: nothing is timed unless the CUDA path equals the oracle on a slice of THIS workload ----
    par = None
    if not args.no_cpu_baseline:
        par = parity_slice(eng, lg, lib_json, asc, asc2, key, kmer, strand, threads, n=args.parity_reads)
        log("[rank %d] parity slice: %s" % (rank, par))

    t0 = time.time()
    packed = eng.pack(asc, pinned=True)
    packed2 = eng.pack(asc2, pinned=True) if asc2 is not None else None
    pack_s = time.time() - t0
    kp = None
    if key is not None:
        kp = eng.pinned_empty(8 * n, np.uint64)
        kp[:] = key
    log("[rank %d] packed %d reads in %.2fs (%.1f Mreads/s host ingest)" % (rank, n, pack_s, n / pack_s / 1e6))

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle import oracle as O
        ns = min(n, args.cpu_sample)
        lo = O.Library(lib_json, k=kmer, strand_filter=strand)
        _ = lo.index
        sec = oracle_pass(O, lo, asc[:ns], None if key is None else key[:ns], threads, None if asc2 is None else asc2[:ns])
        st = oracle_pass.last
        cpu_baseline = {"value": ns / sec, "unit": "reads/s", "cores": threads, "kind": "port",
                        "sample": "first %d reads of the same workload, oracle/nimble_oracle.c: orc_align on %d OpenMP threads (%.2f s), "
                                  "orc_a6_mt on %d threads (%.2f s)" % (ns, threads, st["align_s"], threads, st["a6_s"])}
        log("[cpu] oracle %.0f reads/s on %d threads" % (ns / sec, threads))
    del asc, asc2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    width = lg.config.max_hits_to_report

    class _DevArr:            # wraps a device pointer of the library for torch (zero copy)
        def __init__(self, ptr, n):
            self.__cuda_array_interface__ = {"shape": (int(n),), "typestr": "<i4", "data": (int(ptr), False), "version": 2}

    deferred = world > 1            # multi-GPU: the table's D2H runs beside the NVLink gather (nb200_set_defer_fetch)
    eng.set_defer_fetch(deferred)

    def gather_tables(table):
        """Final count tables -> rank 0, device to device over NVLink (NCCL): one size exchange, then ONE gather of a
        flat int32 buffer [cell | count | feat_off | feat_ids] per rank; this rank's own table goes to its pinned host
        copy (nb200_fetch_counts) WHILE the gather runs.  Returns (device ms, total rows, table)."""
        if world == 1:
            return 0.0, len(table), table
        eng.fetch_counts_start()                     # this rank's D2H starts now, on its own stream, beside everything below
        dv = eng.counts_device()
        parts = [torch.as_tensor(_DevArr(*dv[k_]), device="cuda") for k_ in ("cell", "count", "feat_off", "feat_ids") if dv[k_][1]]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        sizes = torch.zeros(world * 2, dtype=torch.int64, device="cuda")
        mine = torch.tensor([dv["cell"][1], dv["feat_ids"][1]], dtype=torch.int64, device="cuda")
        dist.all_gather_into_tensor(sizes, mine)
        sz = sizes.view(world, 2)
        cap = int((3 * sz[:, 0] + 1 + sz[:, 1]).max().item())
        pad = torch.empty(cap, dtype=torch.int32, device="cuda")
        at = 0
        for p_ in parts:
            pad[at:at + p_.numel()].copy_(p_, non_blocking=True)
            at += p_.numel()
        out = [torch.empty(cap, dtype=torch.int32, device="cuda") for _ in range(world)] if rank == 0 else None
        dist.gather(pad, out, dst=0)                 # asynchronous on NCCL's stream
        table = eng.fetch_counts(copy=False)         # waits for the D2H started above
        e1.record()                                  # recorded after the fetch returned and behind the gather: covers both
        torch.cuda.synchronize()
        assert int(sz[rank, 0].item()) == len(table)
        return e0.elapsed_time(e1), int(sz[:, 0].sum().item()), table

    # ---- device-resident arm: `value` ------------------------------------------------------
    eng.upload(packed, packed2, key=kp)
    table = None
    for _ in range(args.warmup):
        table = eng.align_resident(lg, fetch_counts=not deferred)
        gather_tables(table)
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    dev_ms, wall0 = 0.0, time.perf_counter()
    tim_acc = {}
    gather_ms_acc = []
    for _ in range(args.steps):
        table = eng.align_resident(lg, fetch_counts=not deferred, copy=False)
        t = eng.timing()
        g_ms, total_rows, table = gather_tables(table)
        dev_ms += t["total_ms"] + g_ms
        gather_ms_acc.append(g_ms)
        for k_, v in t.items():
            tim_acc[k_] = tim_acc.get(k_, 0) + v
    barrier()
    wall_ms = 1e3 * (time.perf_counter() - wall0)
    import copy as _copy
    table = _copy.deepcopy(table)           # (a view of the context's pinned table until here)
    ms_per_step = dev_ms / args.steps
    # per-kernel times for the roofline: two more steps with the batch pipelining off (kernels back to back on one
    # stream), because in the pipelined steps above batch k's alignment kernels share the SMs with batch k+1's probe
    eng.set_defer_fetch(False)
    eng.set_overlap(False)
    serial_acc = {}
    for _ in range(2):
        eng.align_resident(lg, fetch_counts=False)
        ts = eng.timing()
        for k_, v in ts.items():
            serial_acc[k_] = serial_acc.get(k_, 0) + v / 2.0
    eng.set_stats(True)                  # device counters of the probe (lookups, sectors): one more untimed pass
    eng.align_resident(lg, fetch_counts=False)
    ts = eng.timing()
    serial_acc["probes"], serial_acc["probe_slots"] = ts["probes"], ts["probe_slots"]
    eng.set_overlap(True)
    eng.set_stats(False)
    # ---- end-to-end arm: host (pinned) buffers in, count table out --------------------------
    eng.set_defer_fetch(deferred)
    for _ in range(2):
        gather_tables(eng.align(lg, packed, packed2, key=kp, fetch_counts=not deferred))
    barrier()
    e2e_wall0 = time.perf_counter()
    for _ in range(args.steps):
        table_e = eng.align(lg, packed, packed2, key=kp, copy=False, fetch_counts=not deferred)      # zero-copy view of the pinned count table
        te = eng.timing()
        _, _, table_e = gather_tables(table_e)
    barrier()
    e2e_ms = 1e3 * (time.perf_counter() - e2e_wall0) / args.steps
    clocks = sampler.stop()                                               # sampled over both timed regions
    same = (np.array_equal(table.cell, table_e.cell) and np.array_equal(table.count, table_e.count)
            and np.array_equal(table.feat_ids, table_e.feat_ids))     # `table` (resident arm) is a copy
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, table, DUMP_BYTES // world, "rank%d_" % rank if world > 1 else "")

    log("[rank %d] resident arm: %.2f ms/step (probe %.2f sw %.2f call %.2f agg %.2f gather %.2f)"
        % (rank, ms_per_step, tim_acc["probe_ms"] / args.steps, tim_acc["sw_ms"] / args.steps, tim_acc["call_ms"] / args.steps,
           tim_acc["agg_ms"] / args.steps, sum(gather_ms_acc) / args.steps))
    stats = torch.tensor([ms_per_step, e2e_ms, wall_ms / args.steps], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
    ms_per_step, e2e_ms, wall_step = (float(x) for x in stats.tolist())
    if rank == 0:
        K = args.steps
        avg = {k_: v / K for k_, v in tim_acc.items()}
        peak, peak_src = peaks()
        pipelined = {"probe": avg["probe_ms"], "sw": avg["sw_ms"], "call": avg["call_ms"], "agg": avg["agg_ms"]}
        avg = dict(avg, probe_ms=serial_acc["probe_ms"], sw_ms=serial_acc["sw_ms"], call_ms=serial_acc["call_ms"],
                   probe_kernel_ms=serial_acc["probe_kernel_ms"], probes=serial_acc["probes"], probe_slots=serial_acc["probe_slots"])
        kern = {"probe": avg["probe_ms"], "probe_kernel": avg["probe_kernel_ms"], "sw": avg["sw_ms"], "call": avg["call_ms"], "agg": avg["agg_ms"],
                "total_serial": serial_acc["total_ms"],
                "note": "each stage timed with the batches serialised (2 extra steps, nb200_set_overlap(0)); in the timed steps "
                        "batch k's sw/call kernels run beside batch k+1's probe, stream-local stage times there: %s"
                        % {k_: round(v, 2) for k_, v in pipelined.items()}}
        dom = max(("probe", "sw", "call", "agg"), key=lambda k_: kern[k_])
        roofline, ra_hbm = probe_roofline(eng, info, avg, n, packed, packed2, width, peak, peak_src, args.workload)
        roofline["dominant_kernel_by_time"] = dom
        dpx_ginst, row_gcups = eng.dpx_peak()
        sw_s = avg["sw_ms"] / 1e3
        gcups = avg["sw_cells"] / sw_s / 1e9 if sw_s > 0 else 0.0
        # DPX instructions the kernel issues: per PAIR of cells (s16x2) one VIADDMNMX.RELU and half a VIMNMX3
        sw_dpx_ginst = avg["sw_cells"] / 2.0 * 1.5 / sw_s / 1e9 if sw_s > 0 else 0.0
        line = {
            "metric": METRIC, "value": world * n / (ms_per_step / 1e3), "unit": "reads/s", "n_gpus": world, "steps": K,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64 k-mers / s16x2 DPX / f64 thresholds", "data": "synthetic",
            "config": make_config(workload, args.workload, n, read_len, kmer, info, world, packed2 is not None),
            "index": {"table_mb": info["table_bytes"] / 1e6, "n_features": info["n_features"]},
            "parity_slice": par,
            "clocks": clocks,
            "e2e": {"value": world * n / (e2e_ms / 1e3), "unit": "reads/s", "h2d_bytes_per_step": int(te["h2d_bytes"]),
                    "d2h_bytes_per_step": int(te["d2h_bytes"]), "ms_per_step": e2e_ms,
                    "api": "nb200_align (C ABI, pinned host buffers in, count table out)",
                    "device_ms": {k_: float(te[k_]) for k_ in ("total_ms", "h2d_ms", "probe_ms", "sw_ms", "call_ms", "agg_ms")}},
            "gpu_launches": int(tim_acc["launches"]),
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
            "kernels_ms_per_step": kern,
            "sw": {"gcups": gcups, "pairs_per_step": avg["sw_pairs"], "cells_per_step": avg["sw_cells"],
                   "candidate_pairs_per_step": avg["sw_items"],
                   "dpx_peak_ginst_per_s": dpx_ginst, "dpx_ginst_per_s": sw_dpx_ginst,
                   "frac_of_dpx_peak": sw_dpx_ginst / dpx_ginst if dpx_ginst else None,
                   "row_recurrence_peak_gcups": row_gcups, "frac_of_row_recurrence_peak": gcups / row_gcups if row_gcups else None,
                   "note": "sw_ms covers window_hash + dedupe + sw_kernel; candidates whose band windows are identical are aligned once. "
                           "dpx peak: register-only VIADDMNMX.S16x2.RELU + VIMNMX3.S16x2 loop (2:1), full occupancy, measured in this run; "
                           "row recurrence peak: the kernel's own row update without memory accesses"},
            "probe": {"lookups_per_read": avg["probes"] / n, "slots_per_lookup": avg["probe_slots"] / max(1.0, avg["probes"]),
                      "glookups_per_s": avg["probes"] / (avg["probe_ms"] / 1e3) / 1e9 if avg["probe_ms"] > 0 else 0.0},
            "gather_ms_per_step": sum(gather_ms_acc) / K,
            "count_rows": int(total_rows), "wall_ms_per_step": wall_step, "resident_equals_e2e": bool(same),
            "host_pack_mreads_per_s": n / pack_s / 1e6,
        }
        if args.workload == "cfg2" and world == 1 and args.hbm_transcripts > 0:
            del packed, kp
            line["roofline_hbm"] = hbm_pass(eng, args, threads, peak, peak_src, ra_hbm)
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
