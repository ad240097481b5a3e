"""C-ABI surface: the shared library loads, exports every symbol include/nimble_b200.h declares,
refuses to run without a GPU (no CPU fallback), and its host-only helpers (packing, host index
build) agree with independent numpy / oracle computations.  No GPU needed."""
import ctypes as ct
import glob
import json
import os
import re

import numpy as np
import pytest

from nimble_b200 import _lib, synth
from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_functions():
    src = open(os.path.join(ROOT, "include", "nimble_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(nb200_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    L = _lib.load()
    declared = header_functions()
    assert len(declared) >= 20
    for name in declared:
        assert hasattr(L, name), "libnimble_b200.so does not export %s" % name
    assert sorted(_lib.EXPORTS) == declared


def test_struct_layouts_match_header():
    assert ct.sizeof(_lib.Config) == 56
    assert ct.sizeof(_lib.Reads) == 56
    assert _lib.RESULT_DTYPE.itemsize == 40 == O.RESULT_DTYPE.itemsize


@pytest.mark.skipif(bool(glob.glob("/dev/nvidia[0-9]*")), reason="a GPU is present")      # any index, not only GPU 0
def test_no_cpu_fallback_without_gpu():
    L = _lib.load()
    ctx = ct.c_void_p()
    rc = L.nb200_create(0, 0, ct.byref(ctx))
    assert rc == _lib.ENODEVICE and not ctx
    assert b"no CPU path" in L.nb200_last_error(None)
    import nimble_b200
    with pytest.raises(nimble_b200.NimbleB200Error):
        nimble_b200.Engine(0)


def numpy_pack(reads, words, stride):
    out = np.zeros((len(reads), stride), np.uint8)
    for i, r in enumerate(reads):
        seq = np.zeros(words, np.uint64)
        nm = np.zeros(words, np.uint32)
        for j, ch in enumerate(r):
            code = "ACGT".find(ch.upper())
            if code < 0:
                nm[j >> 5] |= np.uint32(1 << (j & 31))
                code = 0
            seq[j >> 5] |= np.uint64(code << (2 * (j & 31)))
        out[i, :words * 8] = seq.view(np.uint8)
        out[i, words * 8:words * 12] = nm.view(np.uint8)
    return out


def test_pack_reads_matches_numpy_reference():
    L = _lib.load()
    rng = np.random.default_rng(3)
    reads = ["".join(rng.choice(list("ACGTNacgt"), size=int(n))) for n in rng.integers(0, 151, size=300)]
    reads += ["", "A", "N" * 40, "ACGT" * 37 + "AC"]
    words, stride = ct.c_uint32(), ct.c_uint32()
    assert L.nb200_pack_layout(150, ct.byref(words), ct.byref(stride)) == 0
    assert (words.value, stride.value) == (5, 64)
    off = np.zeros(len(reads) + 1, np.int64)
    np.cumsum([len(r) for r in reads], out=off[1:])
    buf = np.frombuffer("".join(reads).encode(), np.uint8)
    out = np.zeros(len(reads) * stride.value, np.uint8)
    ln = np.zeros(len(reads), np.uint16)
    assert L.nb200_pack_reads(None, buf.ctypes.data, off.ctypes.data, len(reads), words.value, stride.value,
                              out.ctypes.data, ln.ctypes.data) == 0
    assert np.array_equal(ln, [len(r) for r in reads])
    assert np.array_equal(out.reshape(len(reads), -1), numpy_pack(reads, words.value, stride.value))


def test_pack_reads_compact_matches_full_form():
    """Compact wire form == the seq words of the full records; the side table lists exactly the reads with a
    non-ACGT base, ascending, with their N masks (many threads: 6000 reads are split over the host threads)."""
    L = _lib.load()
    rng = np.random.default_rng(5)
    reads = ["".join(rng.choice(list("ACGT"), size=int(n))) for n in rng.integers(0, 151, size=6000)]
    for i in rng.choice(len(reads), size=200, replace=False):
        r = list(reads[i] or "A")
        for j in rng.integers(0, len(r), size=2):
            r[j] = "N" if rng.random() < 0.7 else "x"
        reads[i] = "".join(r)
    words, stride = 5, 64
    off = np.zeros(len(reads) + 1, np.int64)
    np.cumsum([len(r) for r in reads], out=off[1:])
    buf = np.frombuffer("".join(reads).encode(), np.uint8)
    n = len(reads)
    full = np.zeros(n * stride, np.uint8)
    ln = np.zeros(n, np.uint16)
    assert L.nb200_pack_reads(None, buf.ctypes.data, off.ctypes.data, n, words, stride, full.ctypes.data, ln.ctypes.data) == 0
    full = full.reshape(n, stride)
    comp = np.zeros(n * 8 * words, np.uint8)
    ln2 = np.zeros(n, np.uint16)
    need = ct.c_uint64()
    # a table that is too small: NB200_ELIMIT and the size it takes
    idx = np.zeros(10, np.uint32); mask = np.zeros(10 * words, np.uint32)
    rc = L.nb200_pack_reads_compact(None, buf.ctypes.data, off.ctypes.data, n, words, comp.ctypes.data, ln2.ctypes.data,
                                    idx.ctypes.data, mask.ctypes.data, 10, ct.byref(need))
    assert rc == _lib.ELIMIT and need.value == 200
    idx = np.zeros(200, np.uint32); mask = np.zeros(200 * words, np.uint32)
    rc = L.nb200_pack_reads_compact(None, buf.ctypes.data, off.ctypes.data, n, words, comp.ctypes.data, ln2.ctypes.data,
                                    idx.ctypes.data, mask.ctypes.data, 200, ct.byref(need))
    assert rc == 0 and need.value == 200
    assert np.array_equal(ln, ln2)
    assert np.array_equal(comp.reshape(n, 8 * words), full[:, :8 * words])
    nm = full[:, 8 * words:12 * words].copy().view(np.uint32)
    with_n = np.nonzero(nm.any(axis=1))[0]
    assert np.array_equal(idx, with_n.astype(np.uint32))
    assert np.array_equal(mask.reshape(200, words), nm[with_n])


def test_pack_layout_limits():
    L = _lib.load()
    w, s = ct.c_uint32(), ct.c_uint32()
    assert L.nb200_pack_layout(90, ct.byref(w), ct.byref(s)) == 0 and (w.value, s.value) == (3, 48)
    assert L.nb200_pack_layout(500, ct.byref(w), ct.byref(s)) == 0 and w.value == 16
    assert L.nb200_pack_layout(501, ct.byref(w), ct.byref(s)) == _lib.EINVAL
    # a read longer than the layout is an error, not a truncation
    off = np.array([0, 100], np.int64)
    buf = np.frombuffer(b"A" * 100, np.uint8)
    out = np.zeros(48, np.uint8)
    ln = np.zeros(1, np.uint16)
    assert L.nb200_pack_reads(None, buf.ctypes.data, off.ctypes.data, 1, 3, 48, out.ctypes.data, ln.ctypes.data) == _lib.EINVAL


def test_pack_barcodes():
    L = _lib.load()
    cbs = [b"ACGTACGTACGTACGT", b"TTTTTTTTTTTTTTTT", b"ACGTNCGTACGTACGT", b"AAAAAAAAAAAAAAAA"]
    ubs = [b"ACGTACGTACGT", b"GGGGGGGGGGGG", b"ACGTACGTACGT", b"AAAAAAAAAAAC"]
    cb = np.frombuffer(b"".join(cbs), np.uint8)
    ub = np.frombuffer(b"".join(ubs), np.uint8)
    out = np.zeros(4, np.uint64)
    assert L.nb200_pack_barcodes(cb.ctypes.data, 16, ub.ctypes.data, 12, 4, out.ctypes.data) == 0

    def enc(s):
        v = 0
        for ch in s.decode():
            v = (v << 2) | "ACGT".index(ch)
        return v
    assert int(out[0]) == (enc(cbs[0]) << 32) | enc(ubs[0])
    assert int(out[1]) == (0xFFFFFFFF << 32) | enc(ubs[1])
    assert out[2] == _lib.NO_BARCODE
    assert int(out[3]) == 1
    assert synth.unpack_barcode(int(out[0]) >> 32, 16) == cbs[0].decode()


def host_stats(lib_obj, tmp_path, k=20, strand=b"unstranded"):
    L = _lib.load()
    p = tmp_path / "lib.json"
    p.write_text(json.dumps(lib_obj, indent=2))
    out = (ct.c_int64 * 6)()
    rc = L.nb200_host_index_stats(str(p).encode(), strand, k, out)
    return rc, list(out), L.nb200_last_error(None)


@pytest.mark.parametrize("k", [12, 20, 31, 32])
def test_host_index_matches_oracle_index(tmp_path, k):
    lib, _ = synth.allele_family_library(n_founders=5, alleles_per_founder=9, length=500, snps_mean=7, seed=40 + k)
    rc, st, _ = host_stats(lib, tmp_path, k)
    assert rc == 0
    lo = O.Library(lib, k=k)
    assert st[0] == 45 and st[1] == 45 and st[5] == 1
    assert st[2] == lo.index.n_kmers and st[3] == lo.index.n_classes
    assert 4 * st[2] <= st[4] <= 4 * st[2] + 8                        # table entries: load factor 0.25 for small tables (bucketed cuckoo, 2 x 16 B per sector)


def test_host_index_group_on_and_errors(tmp_path):
    lib, _ = synth.allele_family_library(n_founders=3, alleles_per_founder=4, length=300, seed=7, extra_columns=True,
                                         config={"group_on": "gene"})
    rc, st, _ = host_stats(lib, tmp_path)
    assert rc == 0 and st[0] == 12 and st[1] == 3 and st[5] == 0
    rc, _, err = host_stats(lib, tmp_path, k=33)
    assert rc == _lib.EINVAL and b"k must be" in err
    rc, _, err = host_stats(lib, tmp_path, strand=b"sideways")
    assert rc == _lib.EINVAL
    bad = [lib[0], {"headers": ["sequence_name"], "columns": [["a"]]}]
    rc, _, err = host_stats(bad, tmp_path)
    assert rc == _lib.EINVAL and b"sequence" in err
    lib2 = json.loads(json.dumps(lib))
    lib2[1]["columns"][lib2[1]["headers"].index("gene")][0] = "has,comma"
    rc, _, err = host_stats(lib2, tmp_path)
    assert rc == _lib.EINVAL and b"feature name" in err
    (tmp_path / "broken.json").write_text("[{]")
    out = (ct.c_int64 * 6)()
    assert _lib.load().nb200_host_index_stats(str(tmp_path / "broken.json").encode(), b"unstranded", 20, out) == _lib.EINVAL


def test_host_index_beyond_8192_references(tmp_path):
    """Sparse class records: no dense-bitset limit any more."""
    n = 9000
    rng = np.random.default_rng(4)
    seqs = ["".join(rng.choice(list("ACGT"), size=60)) for _ in range(n)]
    lib = [dict(synth.DEFAULT_CONFIG), {"headers": ["reference_genome", "sequence_name", "nt_length", "sequence"],
                                        "columns": [["x"] * n, ["s%05d" % i for i in range(n)], ["60"] * n, seqs]}]
    rc, st, err = host_stats(lib, tmp_path)
    assert rc == 0 and st[0] == n and st[1] == n and st[2] > n * 40


@pytest.mark.parametrize("lf", [None, "0.8", "0.93"])
def test_host_table_self_check_dense_dual_palindromes(tmp_path, lf, monkeypatch):
    """nb200_host_index_stats builds the k-mer table and then looks every library k-mer up through host_lookup (the
    protocol probe_lookup follows on the GPU: first bucket, spill bit, second bucket; own-strand / rc / dual entries),
    in both read orientations, plus one random absent k-mer per key.  Here on a library that holds half of its
    sequences on both strands (dual entries), with dense tables (long cuckoo displacement chains, spilled keys)."""
    if lf:
        monkeypatch.setenv("NB200_TABLE_LF", lf)
    lib, _ = synth.random_transcript_library(n_seqs=300, mean_len=1200, family_frac=0.4, seed=77)
    cols = lib[1]["columns"]
    comp = str.maketrans("ACGT", "TGCA")
    for i in range(0, 300, 2):
        s = cols[3][i].translate(comp)[::-1]
        cols[0].append(cols[0][i]); cols[1].append(cols[1][i] + "_rc"); cols[2].append(str(len(s))); cols[3].append(s)
    for k in (8, 21, 32):
        rc, st, err = host_stats(lib, tmp_path, k)
        assert rc == 0, err
        assert st[0] == 450 and st[4] >= st[2] // 2
    pal = [lib[0], {"headers": lib[1]["headers"], "columns": [["g"] * 2, ["p1", "p2"], ["24", "30"],
                                                                ["ACGTACGTACGTACGTACGTACGT", "AATTAATTAATTAATTGGCCGGCCAATTAA"]]}]
    for k in (4, 8, 12):
        rc, st, err = host_stats(pal, tmp_path, k)
        assert rc == 0, err
