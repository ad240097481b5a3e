"""Python host side above the C ABI (include/nimble_b200.h): device context, library handles,
read packing and the hot-path calls.  Mirrors what nimble's `align()` hands to the aligner
(nimble/__main__.py:153-211) and what `report()` computes (nimble/__main__.py:254-293)."""
from __future__ import annotations

import ctypes as ct
import json
import os
import tempfile
from dataclasses import dataclass

import numpy as np

from . import _lib
from ._lib import CbStats, Config, Counts, NimbleB200Error, Reads, RESULT_DTYPE, Timing


@dataclass
class PackedReads:
    packed: np.ndarray     # uint8 [n * stride]
    length: np.ndarray     # uint16 [n]
    n: int
    stride: int
    words: int
    _keep: object = None
    n_idx: np.ndarray = None   # compact wire form (stride == 8 * words): reads with a non-ACGT base, ascending
    n_mask: np.ndarray = None  # uint32 [len(n_idx) * words]

    def struct(self):
        s = Reads(self.packed.ctypes.data, self.length.ctypes.data, self.n, self.stride, self.words, None, None, 0)
        if self.n_idx is not None and len(self.n_idx):
            s.n_idx, s.n_mask, s.n_with_n = self.n_idx.ctypes.data, self.n_mask.ctypes.data, len(self.n_idx)
        return s

    @property
    def compact(self):
        return self.stride == 8 * self.words

    @property
    def device_stride(self):
        """Bytes per record once on the device (compact records are expanded there)."""
        return (12 * self.words + 15) & ~15

    @property
    def nbytes(self):
        side = 0 if self.n_idx is None else len(self.n_idx) * 4 * (1 + self.words)
        return self.n * (self.stride + 2) + side


@dataclass
class CountTable:
    cell: np.ndarray        # uint32
    count: np.ndarray       # uint32
    feat_off: np.ndarray    # uint32 [n+1]
    feat_ids: np.ndarray    # uint32
    dropped_empty: int
    n_called: int
    n_umis: int
    umis_corrected: int = 0   # (cell, UMI) keys corrected (umi_counts with correct_umis=True)

    def __len__(self):
        return len(self.cell)

    def rows(self, feature_names, cell_name=None):
        """[(feature_string, count, cell)] in the reference's TSV order (nimble/__main__.py:289-293)."""
        out = []
        for i in range(len(self.cell)):
            f = ",".join(feature_names[j] for j in self.feat_ids[self.feat_off[i]:self.feat_off[i + 1]])
            c = int(self.cell[i])
            out.append((f, int(self.count[i]), cell_name(c) if cell_name else c))
        return out


class LibraryHandle:
    def __init__(self, engine, lib_id):
        self.engine = engine
        self.id = lib_id
        self._names = None

    @property
    def info(self):
        v = [ct.c_int64() for _ in range(5)]
        self.engine._ck(self.engine.L.nb200_library_info(self.engine.ctx, self.id, *[ct.byref(x) for x in v]))
        return dict(zip(("n_refs", "n_features", "n_kmers", "n_classes", "table_bytes"), (int(x.value) for x in v)))

    @property
    def config(self):
        c = Config()
        self.engine._ck(self.engine.L.nb200_library_config(self.engine.ctx, self.id, ct.byref(c)))
        return c

    def set_config(self, **kw):
        c = self.config
        for k, v in kw.items():
            if k == "strand_filter" and isinstance(v, str):
                v = _lib.STRAND[v]
            setattr(c, k, v)
        self.engine._ck(self.engine.L.nb200_library_set_config(self.engine.ctx, self.id, ct.byref(c)))

    def set_trim(self, target_length, strictness):
        """`--trim <TARGET_LENGTH>:<STRICTNESS>` for this library (file-level calls; target_length < 0 = off)."""
        self.engine._ck(self.engine.L.nb200_library_set_trim(self.engine.ctx, self.id, int(target_length), float(strictness)))

    @property
    def feature_names(self):
        if self._names is None:
            n = self.info["n_features"]
            self._names = [self.engine.L.nb200_feature_name(self.engine.ctx, self.id, i).decode("utf-8") for i in range(n)]
        return self._names


class Whitelist:
    def __init__(self, engine, wl_id):
        self.engine, self.id = engine, wl_id
        a, b, c, d = ct.c_int64(), ct.c_int64(), ct.c_int64(), ct.c_int32()
        engine._ck(engine.L.nb200_whitelist_info(engine.ctx, wl_id, ct.byref(a), ct.byref(b), ct.byref(c), ct.byref(d)))
        self.n_entries, self.n_unique, self.table_bytes, self.cb_length = a.value, b.value, c.value, d.value

    def entry(self, idx):
        s = self.engine.L.nb200_whitelist_entry(self.engine.ctx, self.id, int(idx))
        return None if s is None else s.decode("latin-1")


class Engine:
    """One CUDA context on one GPU.  Not re-entrant (like the reference: one aligner process)."""

    def __init__(self, device=0, host_threads=0):
        self.L = _lib.load()
        ctx = ct.c_void_p()
        rc = self.L.nb200_create(int(device), int(host_threads), ct.byref(ctx))
        if rc != 0:
            raise NimbleB200Error(rc, (self.L.nb200_last_error(None) or b"").decode())
        self.ctx = ctx
        self._pinned = []

    def close(self):
        if getattr(self, "ctx", None):
            for p in self._pinned:
                self.L.nb200_free_pinned(p)
            self._pinned = []
            self.L.nb200_destroy(self.ctx)
            self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise NimbleB200Error(rc, (self.L.nb200_last_error(self.ctx) or b"").decode())

    # ---- library ---------------------------------------------------------------------------
    def load_library(self, library, strand_filter="unstranded", k=None):
        """library: path to a nimble library JSON or to an index file written by `index` (told apart by its first bytes),
        or the parsed [config, data] object.  k: None = the index file's own k, 20 for a JSON; a k that differs from an
        index file's raises NimbleB200Error."""
        if strand_filter not in _lib.STRAND:
            raise NimbleB200Error(_lib.EINVAL, "unknown --strand_filter value: %r" % (strand_filter,))
        lid = ct.c_int32(-1)
        if isinstance(library, (str, os.PathLike)):
            self._ck(self.L.nb200_load_library(self.ctx, os.fspath(library).encode(), strand_filter.encode(), int(k or 0), ct.byref(lid)))
        else:
            with tempfile.NamedTemporaryFile("w", suffix=".json", delete=False) as f:
                json.dump(library, f)
                path = f.name
            try:
                self._ck(self.L.nb200_load_library(self.ctx, path.encode(), strand_filter.encode(), int(k or 0), ct.byref(lid)))
            finally:
                os.unlink(path)
        return LibraryHandle(self, lid.value)

    def load_feature_names(self, names):
        arr = (ct.c_char_p * max(1, len(names)))(*[n.encode("utf-8") for n in names])
        lid = ct.c_int32(-1)
        self._ck(self.L.nb200_load_feature_names(self.ctx, len(names), arr, ct.byref(lid)))
        return LibraryHandle(self, lid.value)

    # ---- ingest ----------------------------------------------------------------------------
    def pinned_empty(self, nbytes, dtype=np.uint8):
        p = self.L.nb200_alloc_pinned(max(1, int(nbytes)))
        if not p:
            raise NimbleB200Error(_lib.ECUDA, "cudaMallocHost failed")
        self._pinned.append(p)
        buf = (ct.c_uint8 * max(1, int(nbytes))).from_address(p)
        return np.frombuffer(buf, dtype=np.uint8)[:int(nbytes)].view(dtype)

    def pack(self, reads, pinned=True, max_len=None, compact=True):
        """reads: list[str] | uint8 ASCII matrix [n, L] | (uint8 buffer, int64 offsets).
        compact=True (default): the wire form of include/nimble_b200.h — seq words only plus a side table of the
        reads with a non-ACGT base (24 B instead of 48 B per 90-base read across PCIe); False: full records."""
        if isinstance(reads, PackedReads):
            return reads
        if isinstance(reads, np.ndarray) and reads.ndim == 2:
            n, Lr = reads.shape
            buf = np.ascontiguousarray(reads, np.uint8).reshape(-1)
            off = np.arange(0, (n + 1) * Lr, Lr, dtype=np.int64) if Lr else np.zeros(n + 1, np.int64)
        elif isinstance(reads, tuple):
            buf, off = reads
            buf = np.ascontiguousarray(buf, np.uint8)
            off = np.ascontiguousarray(off, np.int64)
            n = len(off) - 1
        else:
            n = len(reads)
            off = np.zeros(n + 1, np.int64)
            if n:
                np.cumsum([len(r) for r in reads], out=off[1:])
            buf = np.frombuffer("".join(reads).encode("ascii", "replace"), np.uint8)
        ml = int((off[1:] - off[:-1]).max()) if n else 1
        if max_len is not None:
            ml = max(ml, int(max_len))
        if ml > _lib.MAX_READ_LEN:
            raise NimbleB200Error(_lib.EINVAL, "read longer than %d bases" % _lib.MAX_READ_LEN)
        words, stride = ct.c_uint32(), ct.c_uint32()
        self._ck(self.L.nb200_pack_layout(max(ml, 1), ct.byref(words), ct.byref(stride)))
        if compact:
            stride.value = 8 * words.value
        nbytes = n * stride.value
        packed = self.pinned_empty(nbytes) if pinned else np.empty(nbytes, np.uint8)
        length = self.pinned_empty(2 * n, np.uint16) if pinned else np.empty(n, np.uint16)
        bp = buf.ctypes.data if len(buf) else off.ctypes.data   # all reads empty: never dereferenced
        if n and not compact:
            self._ck(self.L.nb200_pack_reads(self.ctx, bp, off.ctypes.data, n, words.value, stride.value,
                                             packed.ctypes.data, length.ctypes.data))
        n_idx = n_mask = None
        if n and compact:
            cap, need = n // 64 + 1024, ct.c_uint64(0)
            while True:          # the side table is sized by guess; NB200_ELIMIT reports what it takes
                n_idx = self.pinned_empty(4 * cap, np.uint32) if pinned else np.empty(cap, np.uint32)
                n_mask = self.pinned_empty(4 * cap * words.value, np.uint32) if pinned else np.empty(cap * words.value, np.uint32)
                rc = self.L.nb200_pack_reads_compact(self.ctx, bp, off.ctypes.data, n, words.value, packed.ctypes.data,
                                                     length.ctypes.data, n_idx.ctypes.data, n_mask.ctypes.data, cap, ct.byref(need))
                if rc == _lib.ELIMIT and need.value > cap:
                    cap = int(need.value)
                    continue
                self._ck(rc)
                break
            n_idx, n_mask = n_idx[:need.value], n_mask[:need.value * words.value]
        return PackedReads(packed, length, n, stride.value, words.value, None, n_idx, n_mask)

    def pack_barcodes(self, cb, ub):
        """cb/ub: uint8 ASCII matrices [n, cb_len] / [n, ub_len] -> uint64 keys (cb << 32 | ub)."""
        cb = np.ascontiguousarray(cb, np.uint8)
        ub = np.ascontiguousarray(ub, np.uint8)
        n = cb.shape[0]
        out = np.empty(n, np.uint64)
        rc = self.L.nb200_pack_barcodes(cb.ctypes.data, cb.shape[1], ub.ctypes.data, ub.shape[1], n, out.ctypes.data)
        self._ck(rc)
        return out

    # ---- hot path --------------------------------------------------------------------------
    def _counts(self, c, copy=True):
        """copy=False returns views into the context's pinned count table (valid until the next call)."""
        n = int(c.n_rows)
        def arr(p, m):
            if not m:
                return np.zeros(0, np.uint32)
            a = np.ctypeslib.as_array(p, shape=(m,))
            return a.copy() if copy else a
        off = arr(c.feat_off, n + 1) if n else np.zeros(1, np.uint32)
        return CountTable(arr(c.cell, n), arr(c.count, n), off, arr(c.feat_ids, int(off[-1])),
                          int(c.dropped_empty), int(c.n_called), int(c.n_umis))

    def align(self, lib, r1, r2=None, key=None, threshold=0.05, disable_thresholding=False, per_read=False, copy=True, fetch_counts=True):
        """Host buffers in -> count table out (nb200_align).  per_read=True also returns
        (results[RESULT_DTYPE], feats[n, max_hits])."""
        p1 = self.pack(r1)
        p2 = self.pack(r2) if r2 is not None else None
        s1 = p1.struct()
        s2 = p2.struct() if p2 is not None else None
        kp = None
        if key is not None:
            key = np.ascontiguousarray(key, np.uint64)
            if len(key) != p1.n:
                raise NimbleB200Error(_lib.EINVAL, "key length differs from the number of reads")
            kp = key.ctypes.data
        c = Counts()
        res = feats = None
        rp = fp = None
        if per_read:
            mh = lib.config.max_hits_to_report
            res = np.zeros(p1.n, RESULT_DTYPE)
            feats = np.full((p1.n, mh), -1, np.int32)
            rp, fp = res.ctypes.data, feats.ctypes.data
        self._ck(self.L.nb200_align(self.ctx, lib.id, ct.byref(s1), ct.byref(s2) if s2 is not None else None, kp,
                                    float(threshold), int(bool(disable_thresholding)), rp, fp, ct.byref(c)))
        table = self._counts(c, copy) if fetch_counts else int(c.n_rows)
        return (table, res, feats) if per_read else table

    def upload(self, r1, r2=None, key=None):
        p1 = self.pack(r1)
        p2 = self.pack(r2) if r2 is not None else None
        s1 = p1.struct()
        s2 = p2.struct() if p2 is not None else None
        kp = None
        if key is not None:
            key = np.ascontiguousarray(key, np.uint64)
            kp = key.ctypes.data
        self._ck(self.L.nb200_upload(self.ctx, ct.byref(s1), ct.byref(s2) if s2 is not None else None, kp))
        self._resident_n = p1.n

    def align_resident(self, lib, threshold=0.05, disable_thresholding=False, fetch_counts=True, copy=True):
        c = Counts()
        self._ck(self.L.nb200_align_resident(self.ctx, lib.id, float(threshold), int(bool(disable_thresholding)), ct.byref(c)))
        return self._counts(c, copy) if fetch_counts else int(c.n_rows)

    def align_files(self, inputs, libs, outputs):
        """File-level form (nb200_align_files): FASTQ(.gz) x1-2 or BAM in, one per-read TSV (bulk table for
        FASTQ) per library out, read / parsed / written by the native host code."""
        ins = (ct.c_char_p * len(inputs))(*[os.fspath(p).encode() for p in inputs])
        ids = (ct.c_int32 * len(libs))(*[l.id for l in libs])
        outs = (ct.c_char_p * len(outputs))(*[os.fspath(p).encode() for p in outputs])
        self._ck(self.L.nb200_align_files(self.ctx, ins, len(inputs), ids, outs, len(libs)))

    def align_files_counts(self, inputs, libs, counts_outputs, outputs=None, threshold=0.05, disable_thresholding=False,
                           correct_umis=False):
        """`align` + `report` in one pass (nb200_align_files_counts): BAM with CB/UB tags in, one counts TSV per library
        out (outputs: per-read TSVs written in the same pass, or None).  Returns per library (rows used, count rows,
        dropped UMIs), as report_file does; correct_umis=True (DESIGN.md §2.12) adds the number of UMIs corrected."""
        ins = (ct.c_char_p * len(inputs))(*[os.fspath(p).encode() for p in inputs])
        ids = (ct.c_int32 * len(libs))(*[l.id for l in libs])
        cnt = (ct.c_char_p * len(counts_outputs))(*[os.fspath(p).encode() for p in counts_outputs])
        outs = (ct.c_char_p * len(outputs))(*[os.fspath(p).encode() for p in outputs]) if outputs else None
        w = 4 if correct_umis else 3
        out3 = (ct.c_uint64 * (w * len(libs)))()
        self._ck(self.L.nb200_align_files_counts(self.ctx, ins, len(inputs), ids, outs, cnt, len(libs), float(threshold),
                                                 _lib.umi_flags(disable_thresholding, correct_umis), out3))
        return [tuple(int(v) for v in out3[w * i:w * (i + 1)]) for i in range(len(libs))]

    def report_file(self, in_tsv, out_tsv, threshold=0.05, disable_thresholding=False, correct_umis=False):
        """report() file to file (nb200_report_file).  Returns (rows used, count rows, dropped UMIs), and with
        correct_umis=True (DESIGN.md §2.12) the number of UMIs corrected after them."""
        w = 4 if correct_umis else 3
        out = (ct.c_uint64 * w)()
        self._ck(self.L.nb200_report_file(self.ctx, os.fspath(in_tsv).encode(), os.fspath(out_tsv).encode(), float(threshold),
                                          _lib.umi_flags(disable_thresholding, correct_umis), out))
        return tuple(int(v) for v in out)

    def align_10x_fastq(self, r1_fastq, r2_fastq, whitelist_path, libs, outputs, cb_length=16, umi_length=12):
        """fastq-to-bam + align in one call, no intermediate BAM (nb200_align_10x_fastq).  Returns the barcode statistics."""
        ids = (ct.c_int32 * len(libs))(*[l.id for l in libs])
        outs = (ct.c_char_p * len(outputs))(*[os.fspath(p).encode() for p in outputs])
        st = CbStats()
        self._ck(self.L.nb200_align_10x_fastq(self.ctx, os.fspath(r1_fastq).encode(), os.fspath(r2_fastq).encode(),
                                              os.fspath(whitelist_path).encode(), int(cb_length), int(umi_length), ids, outs,
                                              len(libs), ct.byref(st)))
        return {f: getattr(st, f) for f, _ in CbStats._fields_}

    def fastq_to_counts(self, r1_fastq, r2_fastq, whitelist_path, libs, counts_outputs, cb_length=16, umi_length=12, threshold=0.05,
                        disable_thresholding=False, correct_umis=False):
        """fastq-to-bam + align --counts in one streaming pass, no intermediate BAM (nb200_fastq_to_counts): raw 10x R1 / R2
        in, one counts TSV per library out.  Returns (barcode statistics as fastq_to_bam's, with cache_size 0; per library
        (rows used, count rows, dropped UMIs[, UMIs corrected with correct_umis=True])."""
        ids = (ct.c_int32 * len(libs))(*[l.id for l in libs])
        cnt = (ct.c_char_p * len(counts_outputs))(*[os.fspath(p).encode() for p in counts_outputs])
        w = 4 if correct_umis else 3
        out3 = (ct.c_uint64 * (w * len(libs)))()
        st = CbStats()
        self._ck(self.L.nb200_fastq_to_counts(self.ctx, os.fspath(r1_fastq).encode(), os.fspath(r2_fastq).encode(),
                                              os.fspath(whitelist_path).encode(), int(cb_length), int(umi_length), ids, cnt, len(libs),
                                              float(threshold), _lib.umi_flags(disable_thresholding, correct_umis), out3, ct.byref(st)))
        return ({f: getattr(st, f) for f, _ in CbStats._fields_},
                [tuple(int(v) for v in out3[w * i:w * (i + 1)]) for i in range(len(libs))])

    def set_overlap(self, on):
        """Batch pipelining on (default) / off (kernels back to back on one stream: per-stage times add up)."""
        self._ck(self.L.nb200_set_overlap(self.ctx, int(bool(on))))

    def set_defer_fetch(self, on):
        """Deferred fetch: align / align_resident leave the count table on the device (use fetch_counts=False); fetch_counts()
        copies it into the context's pinned table later, e.g. beside the NCCL gather of the device tables."""
        self._ck(self.L.nb200_set_defer_fetch(self.ctx, int(bool(on))))

    def fetch_counts_start(self):
        """Enqueue the D2H copies of a deferred table and return; fetch_counts() waits for them."""
        self._ck(self.L.nb200_fetch_counts_start(self.ctx))

    def fetch_counts(self, copy=True):
        c = Counts()
        self._ck(self.L.nb200_fetch_counts(self.ctx, ct.byref(c)))
        return self._counts(c, copy)

    def set_stats(self, on):
        """Device counters of the probe (timing()['probes'], ['probe_slots']) on / off (default off)."""
        self._ck(self.L.nb200_set_stats(self.ctx, int(bool(on))))

    def counts_device(self):
        """Device pointers of the last count table: dict name -> (ptr, n_elements) of uint32 arrays
        cell, count, feat_off (n_rows + 1), feat_ids.  For device-to-device gathers (NCCL)."""
        nr, ni = ct.c_uint64(), ct.c_uint64()
        p = [ct.c_void_p() for _ in range(4)]
        self._ck(self.L.nb200_counts_device(self.ctx, ct.byref(nr), ct.byref(ni), *[ct.byref(x) for x in p]))
        n, k = nr.value, ni.value
        return {"cell": (p[0].value or 0, n), "count": (p[1].value or 0, n),
                "feat_off": (p[2].value or 0, n + 1 if n else 0), "feat_ids": (p[3].value or 0, k)}

    def fetch_results(self, lib):
        n = self._resident_n
        mh = lib.config.max_hits_to_report
        res = np.zeros(n, RESULT_DTYPE)
        feats = np.full((n, mh), -1, np.int32)
        self._ck(self.L.nb200_fetch_results(self.ctx, res.ctypes.data, feats.ctypes.data))
        return res, feats

    def umi_counts(self, lib, key, off, feat_ids, score=None, threshold=0.05, disable_thresholding=False, correct_umis=False):
        """report()'s UMI stage on rows (nb200_umi_counts).  correct_umis=True (DESIGN.md §2.12) reads the low half of each
        key as a UMI code (frontend.umi_code) and sets the table's umis_corrected."""
        key = np.ascontiguousarray(key, np.uint64)
        off = np.ascontiguousarray(off, np.uint32)
        feat_ids = np.ascontiguousarray(feat_ids, np.uint32)
        sp = None
        if score is not None:
            score = np.ascontiguousarray(score, np.float64)
            sp = score.ctypes.data
        c = Counts()
        self._ck(self.L.nb200_umi_counts(self.ctx, lib.id, len(key), key.ctypes.data if len(key) else None,
                                         off.ctypes.data, feat_ids.ctypes.data if len(feat_ids) else None, sp,
                                         float(threshold), _lib.umi_flags(disable_thresholding, correct_umis), ct.byref(c)))
        table = self._counts(c)
        n = ct.c_uint64()
        self._ck(self.L.nb200_umis_corrected(self.ctx, ct.byref(n)))
        table.umis_corrected = int(n.value)
        return table

    # ---- fastq-to-bam: cell-barcode correction (nimble/fastq_barcode_processor.py) --------------
    def load_whitelist(self, whitelist, cb_length=16):
        """whitelist: path (one barcode per line, .gz or plain) or a list of str of length cb_length."""
        wid = ct.c_int32()
        if isinstance(whitelist, (str, os.PathLike)):
            self._ck(self.L.nb200_load_whitelist(self.ctx, os.fspath(whitelist).encode(), int(cb_length), ct.byref(wid)))
        else:
            wl = list(whitelist)
            if any(len(w) != cb_length for w in wl):
                raise ValueError("load_whitelist: in-memory entries must all have length cb_length")
            buf = "".join(wl).encode("latin-1")
            self._ck(self.L.nb200_load_whitelist_mem(self.ctx, buf, len(wl), int(cb_length), ct.byref(wid)))
        return Whitelist(self, wid.value)

    @staticmethod
    def _cb_arrays(cb, qual, eligible, L):
        cb = np.ascontiguousarray(cb, np.uint8).reshape(-1, L)
        qual = np.ascontiguousarray(qual, np.uint8).reshape(-1, L)
        if len(cb) != len(qual):
            raise ValueError("cb and qual differ in length")
        el = None if eligible is None else np.ascontiguousarray(eligible, np.uint8)
        return cb, qual, el

    def correct_barcodes(self, wl, cb, qual, eligible=None, out=None):
        """correct_cell_barcode over a batch in file order.  cb, qual: uint8 n x cb_length.
        Returns (idx int32[n] whitelist entry or -1, status uint8[n], stats dict).
        out = (idx, status) preallocated (e.g. pinned) result arrays."""
        cb, qual, el = self._cb_arrays(cb, qual, eligible, wl.cb_length)
        n = len(cb)
        idx, status = out if out is not None else (np.empty(n, np.int32), np.empty(n, np.uint8))
        st = CbStats()
        self._ck(self.L.nb200_correct_barcodes(self.ctx, wl.id, cb.ctypes.data, qual.ctypes.data,
                                               None if el is None else el.ctypes.data, n, idx.ctypes.data,
                                               status.ctypes.data, ct.byref(st)))
        return idx, status, {f: getattr(st, f) for f, _ in CbStats._fields_}

    def cb_upload(self, wl, cb, qual, eligible=None):
        cb, qual, el = self._cb_arrays(cb, qual, eligible, wl.cb_length)
        self._cb_n = len(cb)
        self._ck(self.L.nb200_cb_upload(self.ctx, wl.cb_length, cb.ctypes.data, qual.ctypes.data,
                                        None if el is None else el.ctypes.data, len(cb)))

    def correct_barcodes_resident(self, wl, fetch=True):
        n = self._cb_n
        idx = np.empty(n, np.int32) if fetch else None
        status = np.empty(n, np.uint8) if fetch else None
        st = CbStats()
        self._ck(self.L.nb200_correct_barcodes_resident(self.ctx, wl.id, idx.ctypes.data if fetch else None,
                                                        status.ctypes.data if fetch else None, ct.byref(st)))
        return idx, status, {f: getattr(st, f) for f, _ in CbStats._fields_}

    def fastq_to_bam(self, r1_fastq, r2_fastq, whitelist_path, output_bam, cb_length=16, umi_length=12):
        st = CbStats()
        self._ck(self.L.nb200_fastq_to_bam(self.ctx, os.fspath(r1_fastq).encode(), os.fspath(r2_fastq).encode(),
                                           os.fspath(whitelist_path).encode(), os.fspath(output_bam).encode(),
                                           int(cb_length), int(umi_length), ct.byref(st)))
        return {f: getattr(st, f) for f, _ in CbStats._fields_}

    def random_access_bandwidth(self, nbytes, iters=256):
        """Measured roofline of the probe: (GB/s, Gloads/s) of random 32 B-sector gathers over nbytes."""
        g, l = ct.c_double(), ct.c_double()
        self._ck(self.L.nb200_bench_random_access(self.ctx, int(nbytes), int(iters), ct.byref(g), ct.byref(l)))
        return g.value, l.value

    def dpx_peak(self, iters=4096):
        """Measured integer-pipe ceilings of the Smith-Waterman kernel: (G DPX instructions/s, G cell updates/s of the
        register-only row recurrence)."""
        a, b = ct.c_double(), ct.c_double()
        self._ck(self.L.nb200_bench_dpx_peak(self.ctx, int(iters), ct.byref(a), ct.byref(b)))
        return a.value, b.value

    def timing(self):
        t = Timing()
        self.L.nb200_last_timing(self.ctx, ct.byref(t))
        return {f: getattr(t, f) for f, _ in Timing._fields_}
