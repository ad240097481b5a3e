"""Host-side mirror of nimble's operator interface for the hot path: same function names,
argument meaning and error behaviour as nimble/__main__.py, with the exec of the external aligner
(nimble/__main__.py:195-196) replaced by calls through the C ABI (nimble_b200.engine.Engine).

  generate(file, opt_file, output_path)                         nimble/__main__.py:45-110
  align(reference, output, input, num_cores, strand_filter,
        trim, tmpdir) -> return code                            nimble/__main__.py:153-211
  report(input, output, summarize_columns_list, threshold,
         disable_thresholding)                                  nimble/__main__.py:254-297

File parsing (FASTA/CSV/FASTQ/BAM) is plain Python here — it is outside the timed hot path and is
listed as the next native component in DESIGN.md §7.
"""
from __future__ import annotations

import csv
import gzip
import io
import json
import os
import pathlib
import struct
import sys

import numpy as np

from . import synth


# ---- small utilities restated from nimble/utils.py ------------------------------------------------
def append_path_string(input_path, path_append_string):
    """nimble/utils.py:9-27 — `out.tsv.gz` + `.lib` -> `out.lib.tsv.gz`."""
    filename = os.path.basename(input_path)
    root, ext = filename, ""
    while True:
        root, ext2 = os.path.splitext(root)
        if ext2 == "":
            break
        ext = ext2 + ext
    return os.path.join(os.path.dirname(input_path), root + path_append_string + ext)


def get_library_name_from_filename(seq_path):
    """nimble/utils.py:31-32"""
    return pathlib.Path(seq_path).stem.replace("_", " ")


# ---- generate (nimble/__main__.py:45-110, nimble/parse.py:15-35,78-139) -----------------------------
def _default_config():
    return dict(synth.DEFAULT_CONFIG)      # nimble/types.py:12-25, JSON spelling of Config().__dict__


def parse_fasta(seq_path):
    """nimble/parse.py:15-35 without biopython: id = first word of the header, sequence = joined lines."""
    ref = get_library_name_from_filename(seq_path)
    cols = [[], [], [], []]
    name, chunks = None, []

    def flush():
        if name is not None:
            seq = "".join(chunks)
            cols[0].append(ref)
            cols[1].append(name)      # an empty header gives id "" (biopython's FastaIterator; parse.py:26-29 only maps None to "null")
            cols[2].append(str(len(seq)))
            cols[3].append(seq)
    with open(seq_path) as f:
        for line in f:
            line = line.rstrip("\r\n")
            if line.startswith(">"):
                flush()
                parts = line[1:].split()
                name, chunks = (parts[0] if parts else ""), []
            elif name is not None:
                chunks.append(line.strip())
    flush()
    data = {"headers": ["reference_genome", "sequence_name", "nt_length", "sequence"], "columns": cols}
    return data, _default_config()


def parse_csv(csv_path, has_sequences=True):
    """nimble/parse.py:78-139; `genbank://` sequences need the network and are refused."""
    ref = get_library_name_from_filename(csv_path)
    refs, names, lens, seqs, meta = [], [], [], [], []
    with open(csv_path) as f:
        reader = csv.reader(f, delimiter=",", quotechar='"')
        headers = next(reader)
        sequence_idx = headers.index("sequence") if has_sequences else None
        names_idx = headers.index("name")
        headers.pop(names_idx)
        if has_sequences and names_idx < sequence_idx:
            sequence_idx -= 1
        if has_sequences:
            headers.pop(sequence_idx)
        for row in reader:
            names.append(row.pop(names_idx))
            refs.append(ref)
            if has_sequences:
                raw = row.pop(sequence_idx)
                if "genbank://" in raw:
                    raise ValueError("genbank:// sequences need network access (nimble/remote.py) — not supported")
                seqs.append(raw)
                lens.append(str(len(raw)))
            if not meta:
                meta = [[] for _ in headers]
            for i, col in enumerate(row):
                meta[i].append(col)
    data = {"headers": ["reference_genome", "sequence_name", "nt_length", "sequence"] + headers,
            "columns": [refs, names, lens, seqs] + meta}
    return data, _default_config()


def process_file(file, paired_file):
    data = config = None
    is_csv = False
    if file:
        suffix = pathlib.Path(file).suffix
        if suffix == ".fasta":
            data, config = parse_fasta(file)
        elif suffix == ".csv":
            data, config = parse_csv(file, not paired_file)
            is_csv = True
    return data, config, is_csv


def collate_data(data, metadata):
    """nimble/__main__.py:88-110 — CSV metadata wins, sequences come from the FASTA by name."""
    ni, si, li = (data["headers"].index(h) for h in ("sequence_name", "sequence", "nt_length"))
    mni, msi, mli = (metadata["headers"].index(h) for h in ("sequence_name", "sequence", "nt_length"))
    n = len(data["columns"][si])
    metadata["columns"][msi] = ["" for _ in range(n)]
    metadata["columns"][mli] = ["" for _ in range(n)]
    for from_idx, name in enumerate(data["columns"][ni]):
        if name not in metadata["columns"][mni]:
            print("Error -- record " + name + " is not found in both input files.")
            sys.exit()
        u = metadata["columns"][mni].index(name)
        metadata["columns"][msi][u] = data["columns"][si][from_idx]
        metadata["columns"][mli][u] = data["columns"][li][from_idx]
    return metadata


def generate(file, opt_file, output_path):
    data, config, is_csv_req = process_file(file, opt_file)
    data_opt, config_opt, is_csv_opt = process_file(opt_file, file)
    final_config = config_opt if (data_opt is not None and is_csv_opt) else config
    if data_opt is not None:
        final_data = collate_data(data_opt, data) if is_csv_req else (collate_data(data, data_opt) if is_csv_opt else None)
    else:
        final_data = data
    if final_data is None:
        raise ValueError("generate: --file must end in .fasta or .csv (nimble/__main__.py:76-83)")
    with open(output_path, "w") as f:
        json.dump([final_config, final_data], f, indent=2)


# ---- read ingest ------------------------------------------------------------------------------------
def _open_text(path):
    return gzip.open(path, "rt") if str(path).endswith(".gz") else open(path, "r")


def read_fastq(path):
    names, seqs = [], []
    with _open_text(path) as f:
        while True:
            h = f.readline()
            if not h:
                break
            s = f.readline().rstrip("\r\n")
            f.readline()
            f.readline()
            names.append(h[1:].split()[0] if len(h) > 1 else "")
            seqs.append(s)
    return names, seqs


_BAM_SEQ = "=ACMGRSVTWYHKDBN"


def read_bam(path, want_tags=("CB", "UB", "UR", "GN"), with_qual=False):
    """Minimal BAM reader (BGZF = concatenated gzip members).  Returns per-record tuples:
    (name, flag, sequence, {tag: value}, pos[, qualities as phred+33 text]).  No htslib/pysam needed."""
    with gzip.open(path, "rb") as g:
        buf = g.read()
    if buf[:4] != b"BAM\x01":
        raise ValueError("%s is not a BAM file" % path)
    p = 4
    l_text, = struct.unpack_from("<i", buf, p); p += 4 + l_text
    n_ref, = struct.unpack_from("<i", buf, p); p += 4
    for _ in range(n_ref):
        l_name, = struct.unpack_from("<i", buf, p); p += 4 + l_name + 4
    recs = []
    n = len(buf)
    while p + 4 <= n:
        block_size, = struct.unpack_from("<i", buf, p); p += 4
        end = p + block_size
        (_ref, pos, l_read_name, _mapq, _bin, n_cigar, flag, l_seq, _nref, _npos, _tlen) = struct.unpack_from("<iiBBHHHiiii", buf, p)
        q = p + 32
        name = buf[q:q + l_read_name - 1].decode("ascii", "replace"); q += l_read_name
        q += 4 * n_cigar
        sb = buf[q:q + (l_seq + 1) // 2]; q += (l_seq + 1) // 2
        seq = "".join(_BAM_SEQ[b >> 4] + _BAM_SEQ[b & 15] for b in sb)[:l_seq]
        qual = bytes(b + 33 for b in buf[q:q + l_seq]).decode("ascii") if with_qual else None
        q += l_seq
        tags = {}
        while q + 3 <= end:
            tag = buf[q:q + 2].decode("ascii"); typ = chr(buf[q + 2]); q += 3
            if typ == "Z" or typ == "H":
                e = buf.index(b"\x00", q)
                val = buf[q:e].decode("ascii", "replace"); q = e + 1
            elif typ in "AcC":
                val = buf[q] if typ != "A" else chr(buf[q]); q += 1
            elif typ in "sS":
                val, = struct.unpack_from("<h" if typ == "s" else "<H", buf, q); q += 2
            elif typ in "iI":
                val, = struct.unpack_from("<i" if typ == "i" else "<I", buf, q); q += 4
            elif typ == "f":
                val, = struct.unpack_from("<f", buf, q); q += 4
            elif typ == "B":
                sub = chr(buf[q]); cnt, = struct.unpack_from("<i", buf, q + 1)
                q += 5 + cnt * {"c": 1, "C": 1, "s": 2, "S": 2, "i": 4, "I": 4, "f": 4}[sub]
                val = None
            else:
                raise ValueError("unknown BAM tag type %r" % typ)
            if tag in want_tags:
                tags[tag] = val
        recs.append((name, flag, seq, tags, pos, qual) if with_qual else (name, flag, seq, tags, pos))
        p = end
    return recs


def _revcomp(s):
    return s[::-1].translate(str.maketrans("ACGTNacgtn", "TGCANtgcan"))


def load_reads(inputs):
    """Returns dict(names, r1, r2 or None, cb, ub, extra) from 1-2 FASTQ files or one BAM."""
    ext = os.path.splitext(inputs[0])[-1].lower()
    if ext == ".bam":
        recs = read_bam(inputs[0])
        by_name, order = {}, []
        for name, flag, seq, tags, pos in recs:
            if flag & 0x900:          # secondary / supplementary
                continue
            if flag & 0x10:           # stored reverse-complemented: restore the read as sequenced
                seq = _revcomp(seq)
            slot = by_name.get(name)
            if slot is None:
                slot = by_name[name] = [None, None, {}, {}]
                order.append(name)
            m = 1 if (flag & 0x80) else 0
            slot[m] = seq
            slot[2 + m] = dict(tags, POS=pos + 1 if pos >= 0 else "")   # unaligned records carry no position
        names, r1, r2, cb, ub, extra = [], [], [], [], [], []
        paired = any(v[1] is not None for v in by_name.values())
        for name in order:
            a, b, ta, tb = by_name[name]
            if a is None and b is not None and not paired:
                a, ta = b, tb
            names.append(name); r1.append(a or ""); r2.append(b or "")
            cb.append(ta.get("CB") or ""); ub.append(ta.get("UB") or "")     # UB only: report() keys UMIs on r1_UB and drops rows without it (__main__.py:237-245)
            extra.append((ta, tb))
        return {"names": names, "r1": r1, "r2": r2 if paired else None, "cb": cb, "ub": ub, "extra": extra}
    names, r1 = read_fastq(inputs[0])
    r2 = None
    if len(inputs) > 1:
        _, r2 = read_fastq(inputs[1])
        if len(r2) != len(r1):
            raise ValueError("R1 and R2 FASTQ files hold different numbers of reads")
    return {"names": names, "r1": r1, "r2": r2, "cb": None, "ub": None, "extra": None}


def _string_ids(values):
    """strings -> dense ids in ascending string order ('' -> -1).  Returns (ids, sorted unique)."""
    arr = np.asarray(values, dtype=object)
    uniq = sorted({v for v in values if v})
    idx = {v: i for i, v in enumerate(uniq)}
    return np.array([idx.get(v, -1) for v in arr], np.int64), uniq


_UMI_DIGIT = {"A": 1, "C": 2, "G": 3, "T": 4, "N": 5}
UMI_CODE_MAX = 1525878905          # NNNNNNNNNNNNN
UMI_INTERNED = 0x80000000


def umi_code(umi):
    """The UMI stage's code of a UMI (csrc/umi_code.hpp): an ACGTN string of 1..13 bases is its bijective base-5 value
    (A C G T N = digits 1..5, last base least significant); None for any other string."""
    if not 1 <= len(umi) <= 13:
        return None
    x = 0
    for ch in umi:
        d = _UMI_DIGIT.get(ch)
        if d is None:
            return None
        x = x * 5 + d
    return x


def _umi_ids(values):
    """UMI strings -> the ids nb200_report_file gives them: the code, else the rank among the other UMIs with bit 31 set."""
    codes = [umi_code(v) for v in values]
    other = {v: i for i, v in enumerate(sorted({v for v, c in zip(values, codes) if c is None}))}
    return np.array([c if c is not None else other[v] | UMI_INTERNED for v, c in zip(values, codes)], np.uint64)


def _open_out(path, gz):
    return gzip.open(path, "wt", newline="") if gz else open(path, "w", newline="")


PER_READ_COLUMNS = ["nimble_features", "nimble_score", "r1_forward_score", "r1_reverse_score", "r2_forward_score",
                    "r2_reverse_score", "r1_QNAME", "r1_CB", "r1_UB", "r1_UR", "r1_GN", "r1_POS", "r2_POS"]


def align_10x(reference, output, r1_fastq, r2_fastq, cb_whitelist_file, num_cores=1, strand_filter="unstranded", cb_length=16,
              umi_length=12, k=None, engine=None):
    """`fastq-to-bam` + `align` in one pass over raw 10x FASTQs, without the BAM in between (an extension: the
    reference needs both commands).  Output = the per-read TSV(s) `align` would write for that BAM."""
    from .engine import Engine
    from ._lib import NimbleB200Error
    own = engine is None
    try:
        eng = engine or Engine(int(os.environ.get("LOCAL_RANK", 0)), int(num_cores or 0))
        library_list = reference.split(",")
        outs = [append_path_string(output, "." + os.path.splitext(os.path.basename(l))[0] if len(library_list) > 1 else "")
                for l in library_list]
        libs = [eng.load_library(l, strand_filter=strand_filter, k=k) for l in library_list]
        st = eng.align_10x_fastq(r1_fastq, r2_fastq, cb_whitelist_file, libs, outs, cb_length, umi_length)
        print("nimble_b200: %d pairs, %d with a valid cell barcode (%d corrected) -> %s"
              % (st["total_pairs"], st["written_pairs"], st["cb_corrected"], ", ".join(outs)))
        if own:
            eng.close()
        return 0
    except NimbleB200Error as e:
        print("nimble_b200 aligner error: %s" % e, file=sys.stderr)
        return 1 if e.code != -2 else 2
    except (OSError, ValueError) as e:
        print("nimble_b200 aligner error: %s" % e, file=sys.stderr)
        return 1


def parse_trim(trim, n_libs):
    """`--trim "<TARGET_LENGTH>:<STRICTNESS>[,...]"`, one entry per library (nimble/__main__.py:400) -> [(int, float)] or []."""
    if not trim:
        return []
    out = []
    for item in str(trim).split(","):
        a, sep, b = item.partition(":")
        try:
            t, st = int(a), float(b)
        except ValueError:
            t, st = -1, -1.0
        if not sep or t < 0 or not (0.0 <= st <= 1.0):
            raise ValueError("--trim expects <TARGET_LENGTH>:<STRICTNESS> (strictness 0..1), comma-separated, one entry per library: %r" % (trim,))
        out.append((t, st))
    if len(out) != n_libs:
        raise ValueError("--trim needs one <TARGET_LENGTH>:<STRICTNESS> entry per library")
    return out


def _per_library_paths(path, library_list):
    """nimble/__main__.py:184-189: with several libraries, OUT + "." + library stem (append_path_string)."""
    if path is None:
        return None
    return [append_path_string(path, "." + os.path.splitext(os.path.basename(l))[0] if len(library_list) > 1 else "")
            for l in library_list]


def _print_umi_summary(used, dropped, corrected=None):
    """What `report` prints after writing its counts TSV (nimble/__main__.py:279, write_empty_df); corrected: UMIs merged
    by --correct-umis, printed only when the flag was given."""
    if used == 0:
        print("No data to parse from input file, writing empty output.")
    else:
        if corrected is not None:
            print(f"Corrected {corrected} UMIs (Hamming distance 1)")
        print(f"Dropped {dropped} UMIs due to empty intersections")


def _print_counts_summary(counts_paths, out3):
    """_print_umi_summary per counts file; out3 per library: (rows used, count rows, dropped[, corrected])."""
    for path, o in zip(counts_paths, out3):
        _print_umi_summary(o[0], o[2], o[3] if len(o) > 3 else None)
        print("nimble_b200: wrote %s" % path)


def align_multi_gpu(reference, output, input, num_cores, strand_filter, k, gpus, trim="", counts=None, threshold=0.05,
                    disable_thresholding=False, correct_umis=False):
    """`align` over several GPUs of the node from this one process (nb200_align_files_multi): every library is loaded on
    every GPU, the reader deals slabs of reads to the GPUs, the writer restores input order (outputs byte-identical to a
    one-GPU run).  gpus: a count (devices 0..N-1) or a list of device indices.  counts: the counts TSV path
    (nb200_align_files_counts_multi; output may then be None)."""
    import ctypes as ct
    from . import _lib
    L = _lib.load()
    devs = list(range(int(gpus))) if isinstance(gpus, int) else [int(g) for g in gpus]
    library_list = reference.split(",")
    outs = _per_library_paths(output, library_list)
    cnts = _per_library_paths(counts, library_list)
    d = (ct.c_int32 * len(devs))(*devs)
    ins = (ct.c_char_p * len(input))(*[os.fspath(p).encode() for p in input])
    libs = (ct.c_char_p * len(library_list))(*[os.fspath(p).encode() for p in library_list])
    out_c = (ct.c_char_p * len(outs))(*[os.fspath(p).encode() for p in outs]) if outs else None
    err = ct.create_string_buffer(1024)
    st = (ct.c_double * 4)()
    if cnts is None:
        rc = L.nb200_align_files_multi(d, len(devs), int(num_cores or 0), ins, len(input), libs, len(library_list), strand_filter.encode(), int(k or 0),
                                       out_c, (trim or "").encode(), err, len(err), st)
    else:
        cnt_c = (ct.c_char_p * len(cnts))(*[os.fspath(p).encode() for p in cnts])
        w = 4 if correct_umis else 3
        out3 = (ct.c_uint64 * (w * len(cnts)))()
        rc = L.nb200_align_files_counts_multi(d, len(devs), int(num_cores or 0), ins, len(input), libs, len(library_list), strand_filter.encode(),
                                              int(k or 0), (trim or "").encode(), out_c, cnt_c, float(threshold),
                                              _lib.umi_flags(disable_thresholding, correct_umis), out3, err, len(err), st)
    if rc != 0:
        print("nimble_b200 aligner error: %s" % err.value.decode(errors="replace"), file=sys.stderr)
        return 2 if rc == -2 else 1
    print("nimble_b200: %d reads on %d GPUs in %.2f s (%.1f M reads/s), %d with a feature call" % (st[0], len(devs), st[1], st[0] / max(st[1], 1e-9) / 1e6, st[2]))
    for o in outs or []:
        print("nimble_b200: wrote %s" % o)
    if cnts is not None:
        _print_counts_summary(cnts, [tuple(out3[w * i:w * (i + 1)]) for i in range(len(cnts))])
    return 0


def index(reference, output, k=None, num_cores=0):
    """`index` (extension): build the k-mer index of ONE library JSON on the host (no GPU needed) and save it as an index
    file.  `align`, `fastq-to-counts`, the `aligner` executable and Engine.load_library take that file wherever they take
    the JSON and load it without building the index again.  k: None = 20; num_cores: host threads (0 = all cores).
    Prints k, the reference, feature and k-mer counts and the file size; returns 0, or 1 on an error."""
    from . import _lib
    L = _lib.load()
    rc = L.nb200_index_write(os.fspath(reference).encode(), int(k or 0), int(num_cores or 0), os.fspath(output).encode())
    if rc != 0:
        print("nimble_b200 index error: %s" % (L.nb200_last_error(None) or b"").decode(errors="replace"), file=sys.stderr)
        return 1
    info = index_info(output)
    print("nimble_b200: wrote %s: k = %d, %d references, %d features, %d k-mers, %d bytes"
          % (output, info["k"], info["n_refs"], info["n_features"], info["n_kmers"], os.path.getsize(output)))
    return 0


def index_info(path, verify=False):
    """Header of an index file written by `index` (nb200_index_info) as a dict.  verify=True also checks the device image's
    checksum and looks every k-mer of every reference up in the image read back.  A damaged or foreign file raises
    NimbleB200Error."""
    import ctypes as ct
    from . import _lib
    L = _lib.load()
    out = (ct.c_int64 * 9)()
    rc = L.nb200_index_info(os.fspath(path).encode(), int(bool(verify)), out)
    if rc != 0:
        raise _lib.NimbleB200Error(rc, (L.nb200_last_error(None) or b"").decode(errors="replace"))
    keys = ("version", "k", "n_refs", "n_features", "n_kmers", "n_classes", "n_slots", "identity_features", "image_bytes")
    return dict(zip(keys, (int(v) for v in out)))


def align(reference, output, input, num_cores, strand_filter, trim, tmpdir, k=None, engine=None, native=True, gpus=None, counts=None,
          threshold=0.05, disable_thresholding=False, correct_umis=False):
    """Drop-in for nimble/__main__.py:153-211.  Returns the aligner's return code (0 = success).
    gpus (extension; also $NB200_GPUS): a count or list of devices -> the streaming pipeline over all of them.
    One pass over the reads per library; OUT naming follows __main__.py:184-189.
    native=True (default) hands the files to nb200_align_files (multi-threaded native readers and TSV
    writer, what the `aligner` executable does); native=False keeps file parsing and TSV writing in Python
    around the same GPU calls (the tests use it to cross-check the native file code).
    counts (extension): also write the counts TSV `report` would write from the per-read TSV (threshold /
    disable_thresholding as for report), in the same pass, the rows kept on the GPU; output may then be None (no per-read
    TSV).  Several libraries: one counts file per library, named like the outputs.
    correct_umis (extension, with counts): merge UMIs one substitution away from a better-supported UMI of the same cell
    before the UMI stage (DESIGN.md §2.12)."""
    from .engine import Engine
    from ._lib import NimbleB200Error
    print("Aligning input data to the reference libraries")
    sys.stdout.flush()
    if output is None and counts is None:
        print("nimble_b200 aligner error: align needs --output, --counts or both", file=sys.stderr)
        return 1
    if correct_umis and counts is None:
        print("nimble_b200 aligner error: --correct-umis needs --counts", file=sys.stderr)
        return 1
    if counts is not None and not native:
        print("nimble_b200 aligner error: counts are written by the native file pipeline only (native=True)", file=sys.stderr)
        return 1
    if trim and not native:
        print("nimble_b200: --trim is applied by the native file pipeline only; ignored with native=False")
    if gpus is None and os.environ.get("NB200_GPUS"):
        gpus = int(os.environ["NB200_GPUS"])
    if gpus and engine is None and native and (not isinstance(gpus, int) or gpus > 1):
        return align_multi_gpu(reference, output, list(input), num_cores, strand_filter, k, gpus, trim, counts, threshold, disable_thresholding,
                               correct_umis)
    own = engine is None
    try:
        eng = engine or Engine(int(os.environ.get("LOCAL_RANK", 0)), int(num_cores or 0))
        if native:
            library_list = reference.split(",")
            outs = _per_library_paths(output, library_list)
            cnts = _per_library_paths(counts, library_list)
            trims = parse_trim(trim, len(library_list))
            libs = [eng.load_library(l, strand_filter=strand_filter, k=k) for l in library_list]
            for lg, (t_len, t_strict) in zip(libs, trims):
                lg.set_trim(t_len, t_strict)
            if cnts is None:
                eng.align_files(list(input), libs, outs)
            else:
                out3 = eng.align_files_counts(list(input), libs, cnts, outs, threshold, disable_thresholding, correct_umis)
            for o in outs or []:
                print("nimble_b200: wrote %s" % o)
            if cnts is not None:
                _print_counts_summary(cnts, out3)
            if own:
                eng.close()
            return 0
        data = load_reads(list(input))
        n = len(data["r1"])
        p1 = eng.pack(data["r1"])
        p2 = eng.pack(data["r2"]) if data["r2"] is not None else None
        key = None
        cbs = ubs = None
        if data["cb"] is not None:
            cid, cbs = _string_ids(data["cb"])
            uid, ubs = _string_ids(data["ub"])
            key = ((cid.astype(np.uint64) << np.uint64(32)) | (uid.astype(np.uint64) & np.uint64(0xFFFFFFFF)))
            key[(cid < 0) | (uid < 0)] = np.uint64(0xFFFFFFFFFFFFFFFF)
        library_list = reference.split(",")
        for library in library_list:
            out_append = "." + os.path.splitext(os.path.basename(library))[0] if len(library_list) > 1 else ""
            out_path = append_path_string(output, out_append)
            lg = eng.load_library(library, strand_filter=strand_filter, k=k)
            names = lg.feature_names
            table, res, feats = eng.align(lg, p1, p2, key=key, per_read=True)
            tmp_path = out_path + ".tmp"
            with _open_out(tmp_path, str(out_path).endswith(".gz")) as fh:
                w = csv.writer(fh, delimiter="\t", quoting=csv.QUOTE_NONE, lineterminator="\n", escapechar=None, quotechar=None)
                if key is None:
                    # bulk shape: header, then `<names,comma>\t<count>` (nimble/parse.py:39-57)
                    w.writerow(["nimble_features", "nimble_score"])
                    for f_str, cnt, _cell in table.rows(names):
                        w.writerow([f_str, cnt])
                else:
                    w.writerow(PER_READ_COLUMNS)
                    for i in np.nonzero(res["n_feat"])[0]:
                        ta, tb = data["extra"][i]
                        sc = res["score"][i]
                        w.writerow([",".join(names[j] for j in feats[i, :res["n_feat"][i]]), 1, sc[0], sc[1], sc[2], sc[3],
                                    data["names"][i], data["cb"][i], data["ub"][i], ta.get("UR", ""), ta.get("GN", ""),
                                    ta.get("POS", ""), tb.get("POS", "") if tb else ""])
            os.replace(tmp_path, out_path)
            print("nimble_b200: %d reads, %d called -> %s" % (n, int((res["n_feat"] > 0).sum()) if n else 0, out_path))
        if own:
            eng.close()
        return 0
    except NimbleB200Error as e:
        print("nimble_b200 aligner error: %s" % e, file=sys.stderr)
        return 1 if e.code != -2 else 2
    except (OSError, ValueError) as e:
        print("nimble_b200 aligner error: %s" % e, file=sys.stderr)
        return 1


# ---- report (nimble/__main__.py:213-310) ------------------------------------------------------------------
def write_empty_df(output):
    print("No data to parse from input file, writing empty output.")
    open(output, "w").close()


def report(input, output, summarize_columns_list=None, threshold=0.05, disable_thresholding=False, engine=None, native=True,
           correct_umis=False):
    """Per-read TSV -> counts TSV `feature\\tcount\\tcell_barcode` (no header), UMI stage on the GPU.
    native=True (default): nb200_report_file parses and writes in native code; native=False keeps the TSV
    handling in Python around nb200_umi_counts (the tests cross-check the two).
    correct_umis (extension): merge UMIs one substitution away from a better-supported UMI of the same cell before the
    UMI stage (DESIGN.md §2.12)."""
    from .engine import Engine
    if native:
        own = engine is None
        eng = engine or Engine(int(os.environ.get("LOCAL_RANK", 0)))
        try:
            o = eng.report_file(input, output, threshold, disable_thresholding, correct_umis)
        finally:
            if own:
                eng.close()
        used = o[0]
        _print_umi_summary(used, o[2], o[3] if correct_umis else None)
        if used:
            if summarize_columns_list:
                summarize_fields_tsv(input, summarize_columns_list, "summarize." + output)     # nimble/__main__.py:291-293
        return
    if os.path.getsize(input) == 0:
        write_empty_df(output)
        return
    with _open_text(input) as f:
        reader = csv.reader(f, delimiter="\t", quoting=csv.QUOTE_NONE)
        try:
            header = next(reader)
        except StopIteration:
            write_empty_df(output)
            return
        col = {h: i for i, h in enumerate(header)}
        need = ["nimble_features", "r1_UB", "r1_CB", "nimble_score"]
        for h in need:
            if h not in col:
                raise KeyError(h)
        fi, ui, ci, si = (col[h] for h in need)
        rows = []
        for r in reader:
            if len(r) <= max(fi, ui, ci, si):
                continue
            feats, umi, cb, score = r[fi], r[ui], r[ci], r[si]
            if feats in _PANDAS_NA or umi in _PANDAS_NA or cb in _PANDAS_NA or score in _PANDAS_NA:
                continue
            try:
                s = float(score)
            except ValueError:
                continue
            if s != s:
                continue
            rows.append((cb, umi, feats, s))
    if not rows:
        write_empty_df(output)
        return
    names = sorted({x for r in rows for x in r[2].split(",")})
    fid = {nm: i for i, nm in enumerate(names)}
    cid, cbs = _string_ids([r[0] for r in rows])
    key = (cid.astype(np.uint64) << np.uint64(32)) | _umi_ids([r[1] for r in rows])
    off = np.zeros(len(rows) + 1, np.uint32)
    ids = []
    for i, r in enumerate(rows):
        ids.extend(sorted(fid[x] for x in r[2].split(",")))
        off[i + 1] = len(ids)
    own = engine is None
    eng = engine or Engine(int(os.environ.get("LOCAL_RANK", 0)))
    lib = eng.load_feature_names(names)
    table = eng.umi_counts(lib, key, off, np.array(ids, np.uint32), np.array([r[3] for r in rows], np.float64),
                           threshold, disable_thresholding, correct_umis)
    _print_umi_summary(len(rows), table.dropped_empty, table.umis_corrected if correct_umis else None)
    with open(output, "w", newline="") as f:
        for feat, cnt, cell in table.rows(names):
            f.write("%s\t%d\t%s\n" % (feat, cnt, cbs[cell]))
    if summarize_columns_list:
        summarize_fields_tsv(input, summarize_columns_list, "summarize." + output)     # nimble/__main__.py:291-293
    if own:
        eng.close()


# ---- report --summarize (nimble/__main__.py:295-297) -------------------------------------------------
_PANDAS_NA = {"", "#N/A", "#N/A N/A", "#NA", "-1.#IND", "-1.#QNAN", "-NaN", "-nan", "1.#IND", "1.#QNAN", "<NA>", "N/A",
              "NA", "NULL", "NaN", "None", "n/a", "nan", "null"}


def _infer_column(values):
    """pandas.read_csv type inference for one column of strings: int64 if every cell is an integer,
    float64 if numeric with blanks or decimals, else the strings themselves; NA markers -> None."""
    cells = [None if v in _PANDAS_NA else v for v in values]
    present = [v for v in cells if v is not None]
    try:
        ints = [int(v) for v in present]
        if all(v.strip() == v and "_" not in v for v in present):
            if len(present) == len(cells):
                return [int(v) for v in cells]
            return [None if v is None else float(int(v)) for v in cells]
        del ints
    except ValueError:
        pass
    try:
        if any("_" in v for v in present):
            raise ValueError
        floats = {v: float(v) for v in present}
        return [None if v is None else floats[v] for v in cells]
    except ValueError:
        return cells


def summarize_fields_tsv(input, columns, output_file):
    """summarize_fields on the per-read TSV: per UMI and column, the distinct values with their counts,
    most frequent first (`value(count); ...`), one row per UMI in ascending order."""
    with _open_text(input) as f:
        reader = csv.reader(f, delimiter="\t", quoting=csv.QUOTE_NONE)
        header = next(reader)
        rows = [r + [""] * (len(header) - len(r)) for r in reader]
    rename = {"r1_CB": "cb", "r1_UB": "umi", "nimble_features": "features"}       # convert_df_to_proper_umi :237
    names = [rename.get(h, h) for h in header]
    columns = [rename.get(c, c) for c in columns]
    col = {h: i for i, h in enumerate(names)}
    for c in ["umi"] + list(columns):
        if c not in col:
            raise KeyError(c)
    data = {c: _infer_column([r[col[c]] for r in rows]) for c in set(["umi"] + list(columns))}
    groups = {}
    for i, u in enumerate(data["umi"]):
        if u is not None:
            groups.setdefault(u, []).append(i)

    def fmt(v):
        return repr(v) if isinstance(v, float) else str(v)

    def cell(text):
        # csv.QUOTE_MINIMAL as pandas.to_csv applies it
        if any(ch in text for ch in '\t"\r\n'):
            return '"' + text.replace('"', '""') + '"'
        return text

    with open(output_file, "w", newline="") as f:
        f.write("\t".join(cell(c) for c in ["umi"] + list(columns)) + "\n")
        for u in sorted(groups):
            out = [fmt(u)]
            for c in columns:
                counts = {}
                for i in groups[u]:
                    v = data[c][i]
                    if v is not None:
                        counts[v] = counts.get(v, 0) + 1
                ordered = sorted(counts.items(), key=lambda kv: -kv[1])             # stable: ties keep first appearance
                out.append("; ".join("%s(%d)" % (fmt(k), n) for k, n in ordered))
            f.write("\t".join(cell(x) for x in out) + "\n")


# ---- fastq-to-bam (nimble/fastq_barcode_processor.py:212-316) ----------------------------------------
def fastq_to_bam_with_barcodes(r1_fastq, r2_fastq, cb_whitelist_file, output_bam, num_cores=1, cb_length=16,
                               umi_length=12, engine=None):
    """Paired 10x FASTQ(.gz) + whitelist -> unaligned BAM with CB (corrected) / UB (raw) tags.
    Same signature and console report as the reference; the correction runs on the GPU
    (nb200_fastq_to_bam).  `num_cores` sizes the host parse/compress threads."""
    from .engine import Engine
    from ._lib import NimbleB200Error
    own = engine is None
    eng = engine or Engine(int(os.environ.get("LOCAL_RANK", 0)), host_threads=max(1, int(num_cores)))
    print("Loading cell barcode whitelist...")
    print(f"Processing paired FASTQ files with {num_cores} threads...")
    try:
        st = eng.fastq_to_bam(r1_fastq, r2_fastq, cb_whitelist_file, output_bam, cb_length, umi_length)
    except NimbleB200Error as e:
        print(f"Error during processing: {e}", file=sys.stderr)
        sys.exit(1)
    finally:
        if own:
            eng.close()
    _print_pair_stats(st)
    print(f"\nCorrection cache size: {st['cache_size']} unique raw CBs")
    print(f"\nOutput BAM written to: {output_bam}")
    return st


def _print_pair_stats(st):
    """fastq_to_bam_with_barcodes' statistics (nimble/fastq_barcode_processor.py:284-309) up to the cache size."""
    print("\n=== Processing Statistics ===")
    print(f"Total read pairs: {st['total_pairs']}")
    print(f"Written pairs: {st['written_pairs']}")
    print("\nCell Barcode Correction:")
    print(f"  Perfect matches: {st['cb_perfect_match']}")
    print(f"  Corrected (1-edit): {st['cb_corrected']}")
    print(f"  No valid correction: {st['cb_no_correction']}")
    total = st['cb_perfect_match'] + st['cb_corrected'] + st['cb_no_correction']
    if total > 0:
        print("  Correction rate: %.2f%% perfect, %.2f%% corrected, %.2f%% dropped"
              % (100.0 * st['cb_perfect_match'] / total, 100.0 * st['cb_corrected'] / total,
                 100.0 * st['cb_no_correction'] / total))
    print("\nOther filters:")
    print(f"  Name mismatch: {st['name_mismatch']}")
    print(f"  Too short: {st['too_short']}")
    print(f"  No remaining sequence: {st['no_remaining_seq']}")


def fastq_to_counts(reference, r1_fastq, r2_fastq, cb_whitelist_file, counts, num_cores=1, strand_filter="unstranded", trim="",
                    k=None, gpus=None, cb_length=16, umi_length=12, threshold=0.05, disable_thresholding=False, engine=None,
                    correct_umis=False):
    """`fastq-to-bam`, then `align --counts` on its BAM, in one streaming pass without the BAM (an extension: the reference
    needs fastq-to-bam, align and report).  Raw 10x R1 / R2 FASTQ(.gz) + whitelist in, the counts TSV `report` would
    write out, one per library (named like align's outputs).  gpus (also $NB200_GPUS): a count or a list of devices.
    correct_umis (extension): merge UMIs one substitution away from a better-supported UMI of the same cell before the UMI
    stage (DESIGN.md §2.12).  Returns 0 on success, 1 on an error (with a message on stderr), 2 without a CUDA device."""
    import ctypes as ct
    from . import _lib
    from .engine import Engine
    from ._lib import NimbleB200Error
    library_list = reference.split(",")
    cnts = _per_library_paths(counts, library_list)
    if gpus is None and os.environ.get("NB200_GPUS"):
        gpus = int(os.environ["NB200_GPUS"])
    own = engine is None
    try:
        trims = parse_trim(trim, len(library_list))
        if gpus and engine is None and (not isinstance(gpus, int) or gpus > 1):
            L = _lib.load()
            devs = list(range(int(gpus))) if isinstance(gpus, int) else [int(g) for g in gpus]
            d = (ct.c_int32 * len(devs))(*devs)
            libs = (ct.c_char_p * len(library_list))(*[os.fspath(p).encode() for p in library_list])
            cnt_c = (ct.c_char_p * len(cnts))(*[os.fspath(p).encode() for p in cnts])
            w = 4 if correct_umis else 3
            out3 = (ct.c_uint64 * (w * len(cnts)))()
            cst = _lib.CbStats()
            err = ct.create_string_buffer(1024)
            st4 = (ct.c_double * 4)()
            rc = L.nb200_fastq_to_counts_multi(d, len(devs), int(num_cores or 0), os.fspath(r1_fastq).encode(), os.fspath(r2_fastq).encode(),
                                               os.fspath(cb_whitelist_file).encode(), int(cb_length), int(umi_length), libs, len(library_list),
                                               strand_filter.encode(), int(k or 0), (trim or "").encode(), cnt_c, float(threshold),
                                               _lib.umi_flags(disable_thresholding, correct_umis), out3, ct.byref(cst), err, len(err), st4)
            if rc != 0:
                print("nimble_b200 aligner error: %s" % err.value.decode(errors="replace"), file=sys.stderr)
                return 2 if rc == -2 else 1
            st = {f: getattr(cst, f) for f, _ in _lib.CbStats._fields_}
            o3 = [tuple(out3[w * i:w * (i + 1)]) for i in range(len(cnts))]
        else:
            eng = engine or Engine(int(os.environ.get("LOCAL_RANK", 0)), int(num_cores or 0))
            try:
                libs = [eng.load_library(l, strand_filter=strand_filter, k=k) for l in library_list]
                for lg, (t_len, t_strict) in zip(libs, trims):
                    lg.set_trim(t_len, t_strict)
                st, o3 = eng.fastq_to_counts(r1_fastq, r2_fastq, cb_whitelist_file, libs, cnts, cb_length, umi_length, threshold,
                                             disable_thresholding, correct_umis)
            finally:
                if own:
                    eng.close()
    except NimbleB200Error as e:
        print("nimble_b200 aligner error: %s" % e, file=sys.stderr)
        return 1 if e.code != -2 else 2
    except (OSError, ValueError) as e:
        print("nimble_b200 aligner error: %s" % e, file=sys.stderr)
        return 1
    _print_pair_stats(st)
    if st["no_remaining_seq"] and st["cb_perfect_match"] + st["cb_corrected"] + st["cb_no_correction"] == 0:
        print("nimble_b200: no pair written: every R1 that passed the name and length checks is exactly --cb-length + --umi-length "
              "(%d) bases long, so no read 1 is left after the barcode and UMI (fastq-to-bam drops such pairs)"
              % (int(cb_length) + int(umi_length)), file=sys.stderr)
    _print_counts_summary(cnts, o3)
    return 0
