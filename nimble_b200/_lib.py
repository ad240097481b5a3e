"""ctypes binding of include/nimble_b200.h.  The library is the product: if it is missing or no
CUDA device is present this module raises — there is no CPU fallback."""
from __future__ import annotations

import ctypes as ct
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("NB200_LIB") or os.path.join(HERE, "libnimble_b200.so")   # NB200_LIB: a differently tuned build of the same library

OK, EINVAL, ENODEVICE, ECUDA, EIO, ELIMIT = 0, -1, -2, -3, -4, -5
NO_BARCODE = np.uint64(0xFFFFFFFFFFFFFFFF)
MAX_READ_LEN = 500
STRAND = {"unstranded": 0, "fiveprime": 1, "threeprime": 2, "none": 3}

# every symbol include/nimble_b200.h declares (tests check the .so exports all of them)
EXPORTS = [
    "nb200_create", "nb200_destroy", "nb200_last_error", "nb200_version", "nb200_load_library",
    "nb200_load_library_mem", "nb200_library_config", "nb200_library_set_config", "nb200_library_info",
    "nb200_feature_name", "nb200_pack_layout", "nb200_pack_reads", "nb200_pack_reads_compact", "nb200_pack_barcodes", "nb200_alloc_pinned",
    "nb200_free_pinned", "nb200_align", "nb200_upload", "nb200_align_resident", "nb200_fetch_results",
    "nb200_umi_counts", "nb200_load_feature_names", "nb200_last_timing", "nb200_host_index_stats", "nb200_bench_random_access", "nb200_align_files",
    "nb200_load_whitelist", "nb200_load_whitelist_mem", "nb200_whitelist_info", "nb200_whitelist_entry",
    "nb200_correct_barcodes", "nb200_cb_upload", "nb200_correct_barcodes_resident", "nb200_fastq_to_bam",
    "nb200_counts_device", "nb200_host_ingest_stats", "nb200_report_file",
    "nb200_align_10x_fastq", "nb200_set_overlap", "nb200_bench_dpx_peak", "nb200_set_stats", "nb200_align_files_multi",
    "nb200_library_set_trim", "nb200_trim_maxinfo", "nb200_set_defer_fetch", "nb200_fetch_counts", "nb200_fetch_counts_start", "nb200_fast_inflate",
    "nb200_align_files_counts", "nb200_align_files_counts_multi", "nb200_fastq_to_counts", "nb200_fastq_to_counts_multi",
    "nb200_index_write", "nb200_index_info", "nb200_umis_corrected", "nb200_umi_neighbours",
]

# flags word of the counting entries (the disable_thresholding parameter)
UMI_NO_THRESHOLD, UMI_CORRECT = 1, 2


def umi_flags(disable_thresholding, correct_umis):
    return (UMI_NO_THRESHOLD if disable_thresholding else 0) | (UMI_CORRECT if correct_umis else 0)

CB_SKIPPED, CB_PERFECT, CB_CORRECTED, CB_NONE = 0, 1, 2, 3


class Config(ct.Structure):
    _fields_ = [("k", ct.c_int32), ("score_threshold", ct.c_int32), ("score_filter", ct.c_int32),
                ("score_percent", ct.c_double), ("num_mismatches", ct.c_int32),
                ("discard_multiple_matches", ct.c_int32), ("intersect_level", ct.c_int32),
                ("discard_multi_hits", ct.c_int32), ("require_valid_pair", ct.c_int32),
                ("max_hits_to_report", ct.c_int32), ("strand_filter", ct.c_int32), ("pad_", ct.c_int32)]


class Reads(ct.Structure):
    _fields_ = [("packed", ct.c_void_p), ("len", ct.c_void_p), ("n", ct.c_uint64),
                ("stride", ct.c_uint32), ("words", ct.c_uint32),
                ("n_idx", ct.c_void_p), ("n_mask", ct.c_void_p), ("n_with_n", ct.c_uint64)]


class Counts(ct.Structure):
    _fields_ = [("n_rows", ct.c_uint64), ("cell", ct.POINTER(ct.c_uint32)), ("count", ct.POINTER(ct.c_uint32)),
                ("feat_off", ct.POINTER(ct.c_uint32)), ("feat_ids", ct.POINTER(ct.c_uint32)),
                ("dropped_empty", ct.c_uint64), ("n_called", ct.c_uint64), ("n_umis", ct.c_uint64)]


class Timing(ct.Structure):
    _fields_ = [("total_ms", ct.c_float), ("probe_ms", ct.c_float), ("sw_ms", ct.c_float), ("call_ms", ct.c_float),
                ("agg_ms", ct.c_float), ("h2d_ms", ct.c_float), ("probes", ct.c_uint64), ("probe_slots", ct.c_uint64),
                ("sw_pairs", ct.c_uint64), ("sw_cells", ct.c_uint64), ("launches", ct.c_uint64),
                ("h2d_bytes", ct.c_uint64), ("d2h_bytes", ct.c_uint64), ("sw_items", ct.c_uint64),
                ("probe_kernel_ms", ct.c_float), ("pad_", ct.c_float),
                ("probe_warp_reads", ct.c_uint64)]


class CbStats(ct.Structure):
    _fields_ = [(f, ct.c_uint64) for f in ("total_pairs", "written_pairs", "cb_perfect_match", "cb_corrected",
                                           "cb_no_correction", "name_mismatch", "too_short", "no_remaining_seq",
                                           "cache_size", "n_exact_miss", "n_multi", "probes", "launches",
                                           "h2d_bytes", "d2h_bytes")] + [("kernel_ms", ct.c_float), ("total_ms", ct.c_float)]


RESULT_DTYPE = np.dtype([
    ("score", "<u2", (4,)), ("n_hits", "<u2", (4,)), ("n_cand", "<u2", (4,)),
    ("edits", "u1", (4,)), ("status", "u1", (4,)),
    ("reason", "u1"), ("config", "u1"), ("n_feat", "u1"), ("n_sw", "u1"), ("pair_score", "<u4"),
])


class NimbleB200Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("nimble_b200 error %d: %s" % (code, msg))
        self.code = code


_lib = None


def load():
    """Load libnimble_b200.so (built in-tree by nimble_b200/build.py).  Raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise ImportError("nimble_b200: %s is missing — run `python -m nimble_b200.build` (nvcc, sm_100a). "
                          "There is no CPU fallback." % SO_PATH)
    L = ct.CDLL(SO_PATH)
    vp, i32, u32, u64, dbl = ct.c_void_p, ct.c_int32, ct.c_uint32, ct.c_uint64, ct.c_double
    L.nb200_create.argtypes = [i32, i32, ct.POINTER(vp)]
    L.nb200_destroy.argtypes = [vp]
    L.nb200_destroy.restype = None
    L.nb200_last_error.argtypes = [vp]
    L.nb200_last_error.restype = ct.c_char_p
    L.nb200_version.restype = ct.c_char_p
    L.nb200_load_library.argtypes = [vp, ct.c_char_p, ct.c_char_p, i32, ct.POINTER(i32)]
    L.nb200_load_library_mem.argtypes = [vp, i32, ct.POINTER(ct.c_char_p), ct.POINTER(ct.c_char_p),
                                         ct.POINTER(ct.c_char_p), ct.POINTER(Config), ct.POINTER(i32)]
    L.nb200_library_config.argtypes = [vp, i32, ct.POINTER(Config)]
    L.nb200_library_set_config.argtypes = [vp, i32, ct.POINTER(Config)]
    L.nb200_library_info.argtypes = [vp, i32] + [ct.POINTER(ct.c_int64)] * 5
    L.nb200_feature_name.argtypes = [vp, i32, u32]
    L.nb200_feature_name.restype = ct.c_char_p
    L.nb200_pack_layout.argtypes = [u32, ct.POINTER(u32), ct.POINTER(u32)]
    L.nb200_pack_reads.argtypes = [vp, vp, vp, u64, u32, u32, vp, vp]
    L.nb200_pack_reads_compact.argtypes = [vp, vp, vp, u64, u32, vp, vp, vp, vp, u64, ct.POINTER(u64)]
    L.nb200_pack_barcodes.argtypes = [vp, u32, vp, u32, u64, vp]
    L.nb200_alloc_pinned.argtypes = [ct.c_size_t]
    L.nb200_alloc_pinned.restype = vp
    L.nb200_free_pinned.argtypes = [vp]
    L.nb200_free_pinned.restype = None
    L.nb200_align.argtypes = [vp, i32, ct.POINTER(Reads), ct.POINTER(Reads), vp, dbl, i32, vp, vp, ct.POINTER(Counts)]
    L.nb200_upload.argtypes = [vp, ct.POINTER(Reads), ct.POINTER(Reads), vp]
    L.nb200_align_resident.argtypes = [vp, i32, dbl, i32, ct.POINTER(Counts)]
    L.nb200_fetch_results.argtypes = [vp, vp, vp]
    L.nb200_umi_counts.argtypes = [vp, i32, u64, vp, vp, vp, vp, dbl, i32, ct.POINTER(Counts)]
    L.nb200_load_feature_names.argtypes = [vp, i32, ct.POINTER(ct.c_char_p), ct.POINTER(i32)]
    L.nb200_last_timing.argtypes = [vp, ct.POINTER(Timing)]
    L.nb200_align_files.argtypes = [vp, ct.POINTER(ct.c_char_p), i32, ct.POINTER(i32), ct.POINTER(ct.c_char_p), i32]
    L.nb200_bench_random_access.argtypes = [vp, u64, u32, ct.POINTER(dbl), ct.POINTER(dbl)]
    L.nb200_bench_dpx_peak.argtypes = [vp, u32, ct.POINTER(dbl), ct.POINTER(dbl)]
    L.nb200_host_index_stats.argtypes = [ct.c_char_p, ct.c_char_p, i32, ct.POINTER(ct.c_int64)]
    L.nb200_index_write.argtypes = [ct.c_char_p, i32, i32, ct.c_char_p]
    L.nb200_index_info.argtypes = [ct.c_char_p, i32, ct.POINTER(ct.c_int64)]
    L.nb200_align_10x_fastq.argtypes = [vp, ct.c_char_p, ct.c_char_p, ct.c_char_p, i32, i32, ct.POINTER(i32), ct.POINTER(ct.c_char_p), i32,
                                        ct.POINTER(CbStats)]
    L.nb200_set_overlap.argtypes = [vp, i32]
    L.nb200_set_stats.argtypes = [vp, i32]
    L.nb200_set_defer_fetch.argtypes = [vp, i32]
    L.nb200_fetch_counts.argtypes = [vp, ct.POINTER(Counts)]
    L.nb200_fetch_counts_start.argtypes = [vp]
    L.nb200_fast_inflate.argtypes = [vp, u64, vp, u64]
    L.nb200_align_files_multi.argtypes = [ct.POINTER(i32), i32, i32, ct.POINTER(ct.c_char_p), i32, ct.POINTER(ct.c_char_p), i32, ct.c_char_p, i32,
                                          ct.POINTER(ct.c_char_p), ct.c_char_p, ct.c_char_p, ct.c_size_t, ct.POINTER(dbl)]
    L.nb200_align_files_counts.argtypes = [vp, ct.POINTER(ct.c_char_p), i32, ct.POINTER(i32), ct.POINTER(ct.c_char_p), ct.POINTER(ct.c_char_p), i32,
                                           dbl, i32, ct.POINTER(u64)]
    L.nb200_align_files_counts_multi.argtypes = [ct.POINTER(i32), i32, i32, ct.POINTER(ct.c_char_p), i32, ct.POINTER(ct.c_char_p), i32, ct.c_char_p,
                                                 i32, ct.c_char_p, ct.POINTER(ct.c_char_p), ct.POINTER(ct.c_char_p), dbl, i32, ct.POINTER(u64),
                                                 ct.c_char_p, ct.c_size_t, ct.POINTER(dbl)]
    L.nb200_fastq_to_counts.argtypes = [vp, ct.c_char_p, ct.c_char_p, ct.c_char_p, i32, i32, ct.POINTER(i32), ct.POINTER(ct.c_char_p), i32,
                                        dbl, i32, ct.POINTER(u64), ct.POINTER(CbStats)]
    L.nb200_fastq_to_counts_multi.argtypes = [ct.POINTER(i32), i32, i32, ct.c_char_p, ct.c_char_p, ct.c_char_p, i32, i32,
                                              ct.POINTER(ct.c_char_p), i32, ct.c_char_p, i32, ct.c_char_p, ct.POINTER(ct.c_char_p), dbl,
                                              i32, ct.POINTER(u64), ct.POINTER(CbStats), ct.c_char_p, ct.c_size_t, ct.POINTER(dbl)]
    L.nb200_library_set_trim.argtypes = [vp, i32, i32, dbl]
    L.nb200_trim_maxinfo.argtypes = [vp, u32, i32, i32, dbl]
    L.nb200_trim_maxinfo.restype = u32
    L.nb200_report_file.argtypes = [vp, ct.c_char_p, ct.c_char_p, dbl, i32, ct.POINTER(u64)]
    L.nb200_umis_corrected.argtypes = [vp, ct.POINTER(u64)]
    L.nb200_umi_neighbours.argtypes = [u32, ct.POINTER(u32), ct.POINTER(u32)]
    L.nb200_host_ingest_stats.argtypes = [ct.POINTER(ct.c_char_p), i32, i32, ct.POINTER(u64)]
    L.nb200_counts_device.argtypes = [vp, ct.POINTER(u64), ct.POINTER(u64)] + [ct.POINTER(vp)] * 4
    L.nb200_load_whitelist.argtypes = [vp, ct.c_char_p, i32, ct.POINTER(i32)]
    L.nb200_load_whitelist_mem.argtypes = [vp, vp, u64, i32, ct.POINTER(i32)]
    L.nb200_whitelist_info.argtypes = [vp, i32, ct.POINTER(ct.c_int64), ct.POINTER(ct.c_int64), ct.POINTER(ct.c_int64),
                                       ct.POINTER(i32)]
    L.nb200_whitelist_entry.argtypes = [vp, i32, u32]
    L.nb200_whitelist_entry.restype = ct.c_char_p
    L.nb200_correct_barcodes.argtypes = [vp, i32, vp, vp, vp, u64, vp, vp, ct.POINTER(CbStats)]
    L.nb200_cb_upload.argtypes = [vp, i32, vp, vp, vp, u64]
    L.nb200_correct_barcodes_resident.argtypes = [vp, i32, vp, vp, ct.POINTER(CbStats)]
    L.nb200_fastq_to_bam.argtypes = [vp, ct.c_char_p, ct.c_char_p, ct.c_char_p, ct.c_char_p, i32, i32, ct.POINTER(CbStats)]
    for name in EXPORTS:
        f = getattr(L, name)
        if f.restype is ct.c_int:   # default -> int32 status
            f.restype = i32
    assert ct.sizeof(Config) == 56 and RESULT_DTYPE.itemsize == 40 and ct.sizeof(CbStats) == 128
    _lib = L
    return L
