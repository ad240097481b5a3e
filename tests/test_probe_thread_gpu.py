"""Thread-per-read probe (probe_thread_kernel + probe_list_kernel) against the warp-per-read probe that
NB200_PROBE_WARP=1 selects: identical per-read records, feature ids, count tables and probe counters (lookups,
sectors read) on every case, and both bit-exact against the C oracle."""
import os

import numpy as np
import pytest

from nimble_b200 import synth
from oracle import oracle as O
from helpers import diff_results, oracle_counts, table_tuple, to_concat

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def engine():
    """A context that builds libraries on one host thread.  The multi-threaded build places keys in a racy order, so
    two loads of one library may differ in which keys sit in their second bucket, and so in the sectors a probe reads;
    built on one thread, the two loads compared below are the same table and every counter must agree."""
    import nimble_b200
    eng = nimble_b200.Engine(0, host_threads=1)
    yield eng
    eng.close()


def _load(engine, lib, k, env):
    old = {name: os.environ.get(name) for name in env}
    os.environ.update(env)
    try:
        return engine.load_library(lib, k=k)
    finally:
        for name, v in old.items():
            if v is None:
                os.environ.pop(name, None)
            else:
                os.environ[name] = v


def thread_vs_warp(engine, lib, r1, key, k, env=None):
    """Aligns r1 with the thread probe and with the warp probe, device probe counters on; returns the thread run's
    fallback count."""
    lo = O.Library(lib, k=k)
    ro, fo = O.align(lo, to_concat(r1))
    cell, cnt, off, ids, dropped = oracle_counts(lo, ro, fo, key, 0.05)
    runs = []
    engine.set_stats(True)
    try:
        for warp in (False, True):
            e = dict(env or {})
            if warp:
                e["NB200_PROBE_WARP"] = "1"
            lg = _load(engine, lib, k, e)
            table, rg, fg = engine.align(lg, r1, key=key, per_read=True)
            tm = engine.timing()
            bad = diff_results(ro, fo, rg, fg)
            assert not bad, ("warp probe" if warp else "thread probe") + ":\n" + "\n".join(bad)
            tt = table_tuple(table.cell, table.count, table.feat_off, table.feat_ids)
            assert tt == table_tuple(cell, cnt, off, ids) and table.dropped_empty == dropped
            runs.append((rg, fg, tt, tm))
    finally:
        engine.set_stats(False)
    (rt, ft, tt, mt), (rw, fw, tw, mw) = runs
    assert np.array_equal(rt, rw) and np.array_equal(ft, fw) and tt == tw
    # listed reads are counted by probe_list_kernel alone: the counters are those of the warp probe
    assert mt["probes"] > 0 and (mt["probes"], mt["probe_slots"]) == (mw["probes"], mw["probe_slots"])
    assert mw["probe_warp_reads"] == 0       # the warp probe lists nothing
    return mt["probe_warp_reads"]


def test_cfg2_shape(engine):
    lib, codes = synth.allele_family_library(seed=1)
    r1, truth = synth.sample_reads(codes, 80_000, read_len=90, seed=2)
    key = synth.barcodes_10x(len(r1), n_cells=200, seed=2, truth=truth)
    fb = thread_vs_warp(engine, lib, r1, key, k=20)
    assert fb < len(r1) // 10


@pytest.mark.parametrize("lf", [None, "0.95"])
def test_transcripts_k31(engine, lf):
    """k = 31; at load factor 0.95 many keys sit in their second bucket."""
    lib, codes = synth.random_transcript_library(n_seqs=1500, mean_len=1500, family_frac=0.3, seed=5,
                                                 config={"score_percent": 0.25})
    r1, truth = synth.sample_reads(codes, 40_000, read_len=100, rc_frac=0.3, seed=6)
    key = synth.barcodes_10x(len(r1), n_cells=100, seed=6, truth=truth)
    thread_vs_warp(engine, lib, r1, key, k=31, env={"NB200_TABLE_LF": lf} if lf else None)


def test_n_bases_short_and_mixed_lengths(engine):
    """Lengths 1-300 side by side in every warp, N bases anywhere (k-mers that span one are skipped)."""
    lib, codes = synth.allele_family_library(n_founders=8, alleles_per_founder=40, seed=11)
    rng = np.random.default_rng(12)
    acgt = np.frombuffer(b"ACGT", np.uint8)
    reads = []
    for _ in range(12_000):
        L = int(rng.integers(1, 301))
        c = codes[int(rng.integers(0, len(codes)))]
        a = int(rng.integers(0, len(c) - L + 1))
        s = acgt[c[a:a + L]].copy()
        if rng.random() < 0.3:
            s[rng.integers(0, L, size=int(rng.integers(1, 4)))] = ord("N")
        if rng.random() < 0.3:
            s = s[::-1].copy()
            s[s != ord("N")] = acgt[3 - np.searchsorted(acgt, s[s != ord("N")])]
        reads.append(s.tobytes().decode("ascii"))
    key = synth.barcodes_10x(len(reads), n_cells=50, seed=12)
    thread_vs_warp(engine, lib, reads, key, k=20)


def test_dual_records(engine):
    """Every fourth allele also enters the library reverse-complemented: its k-mers are present on both strands."""
    lib, codes = synth.allele_family_library(n_founders=6, alleles_per_founder=30, seed=21)
    cols = lib[1]["columns"]
    acgt = np.frombuffer(b"ACGT", np.uint8)
    extra = [(3 - c[::-1]).astype(np.uint8) for c in codes[::4]]
    for j, c in enumerate(extra):
        cols[0].append(cols[0][0]); cols[1].append("RC-%03d" % j); cols[2].append(str(len(c)))
        cols[3].append(acgt[c].tobytes().decode("ascii"))
    r1, truth = synth.sample_reads(codes + extra, 30_000, read_len=90, rc_frac=0.5, seed=22)
    key = synth.barcodes_10x(len(r1), n_cells=60, seed=22, truth=truth)
    thread_vs_warp(engine, lib, r1, key, k=20)


def test_wide_and_overflow_classes_take_the_list(engine):
    """250 alleles per founder: shared k-mers fall in classes of 8 words (overflow form), so many reads start on a
    class wider than 4 words and only narrow down at their SNPs; those reads go through the warp list."""
    lib, codes = synth.allele_family_library(n_founders=4, alleles_per_founder=250, length=900, snps_mean=8.0, seed=31)
    r1, truth = synth.sample_reads(codes, 30_000, read_len=90, rc_frac=0.3, seed=32)
    key = synth.barcodes_10x(len(r1), n_cells=60, seed=32, truth=truth)
    fb = thread_vs_warp(engine, lib, r1, key, k=20)
    assert 0 < fb < len(r1)


@pytest.mark.parametrize("cap", ["0", "2"])
def test_narrow_cap(engine, cap):
    """A lowered shared-memory list cap also bounds the thread path's anchors (0: every hit read goes wide)."""
    lib, codes = synth.allele_family_library(n_founders=6, alleles_per_founder=60, seed=41)
    r1, truth = synth.sample_reads(codes, 8_000, read_len=90, rc_frac=0.3, seed=42)
    key = synth.barcodes_10x(len(r1), n_cells=30, seed=42, truth=truth)
    fb = thread_vs_warp(engine, lib, r1, key, k=20, env={"NB200_NARROW_CAP": cap})
    assert fb > 0
