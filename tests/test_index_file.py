"""Index files (`python -m nimble_b200 index`, nb200_index_write / nb200_index_info): written and checked on the host
without a GPU.  The header agrees with nb200_host_index_stats, the verify pass accepts the library shapes of
test_abi.py, and damaged or foreign files are refused with a reason."""
import ctypes as ct
import json
import os
import struct

import numpy as np
import pytest

from nimble_b200 import _lib, frontend, synth
from nimble_b200.__main__ import main

# header offsets (library.hpp, IndexHeader)
OFF_VERSION, OFF_N_KMERS, OFF_SECTIONS, OFF_FILE_BYTES, OFF_HEADER_SUM, HEADER_BYTES = 8, 88, 296, 392, 400, 408
SECTIONS = ["feature_names", "tok_end", "tok_comma", "device image"]
C = np.uint64(0x9E3779B97F4A7C15)


def py_checksum(buf, word0=0):
    """checksum.hpp in numpy: sum mod 2^64 of splitmix64(w_i ^ i * C)."""
    b = bytes(buf) + b"\0" * (-len(buf) % 8)
    w = np.frombuffer(b, "<u8")
    with np.errstate(over="ignore"):
        i = np.arange(word0, word0 + len(w), dtype=np.uint64)
        z = (w ^ (i * C)) + C
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
        return int(z.sum(dtype=np.uint64))


def sections(data):
    return [struct.unpack_from("<QQQ", data, OFF_SECTIONS + 24 * s) for s in range(len(SECTIONS))]


def reseal(data):
    """Recompute the header checksum after an edit of the header."""
    data[OFF_HEADER_SUM:OFF_HEADER_SUM + 8] = b"\0" * 8
    struct.pack_into("<Q", data, OFF_HEADER_SUM, py_checksum(data[:HEADER_BYTES]))


def write_json(lib, path):
    path.write_text(json.dumps(lib))
    return path


def write_index(json_path, out, k=20):
    rc = _lib.load().nb200_index_write(str(json_path).encode(), k, 0, str(out).encode())
    return rc, (_lib.load().nb200_last_error(None) or b"").decode()


def info(path, verify=1):
    out = (ct.c_int64 * 9)()
    rc = _lib.load().nb200_index_info(str(path).encode(), verify, out)
    return rc, list(out), (_lib.load().nb200_last_error(None) or b"").decode()


def host_stats(json_path, k):
    out = (ct.c_int64 * 6)()
    assert _lib.load().nb200_host_index_stats(str(json_path).encode(), b"unstranded", k, out) == 0
    return list(out)


def dense_dual_library():
    """test_abi.py's dense transcript shape: half of the sequences also on the other strand (dual entries)."""
    lib, _ = synth.random_transcript_library(n_seqs=300, mean_len=1200, family_frac=0.4, seed=77)
    cols = lib[1]["columns"]
    comp = str.maketrans("ACGT", "TGCA")
    for i in range(0, 300, 2):
        s = cols[3][i].translate(comp)[::-1]
        cols[0].append(cols[0][i]); cols[1].append(cols[1][i] + "_rc"); cols[2].append(str(len(s))); cols[3].append(s)
    return lib


@pytest.fixture
def small_index(tmp_path):
    lib, _ = synth.allele_family_library(n_founders=3, alleles_per_founder=4, length=300, seed=7, extra_columns=True,
                                         config={"group_on": "gene"})
    j = write_json(lib, tmp_path / "lib.json")
    out = tmp_path / "lib.nb200idx"
    assert write_index(j, out)[0] == 0
    return out


def test_index_command_writes_a_file_without_gpu(tmp_path, capsys):
    lib, _ = synth.allele_family_library(n_founders=4, alleles_per_founder=6, length=400, seed=3)
    j = write_json(lib, tmp_path / "lib.json")
    out = tmp_path / "lib.nb200idx"
    with pytest.raises(SystemExit) as e:
        main(["index", "--reference", str(j), "--output", str(out), "-k", "24", "-c", "2"])
    assert e.value.code == 0
    text = capsys.readouterr().out
    st = host_stats(j, 24)
    assert "k = 24, 24 references, 24 features, %d k-mers, %d bytes" % (st[2], os.path.getsize(out)) in text
    assert out.read_bytes()[:8] == b"NB200IDX" and not os.path.exists(str(out) + ".tmp")
    assert frontend.index_info(out, verify=True)["k"] == 24


@pytest.mark.parametrize("k", [12, 20, 31, 32])
def test_index_info_equals_host_index_stats(tmp_path, k):
    lib, _ = synth.allele_family_library(n_founders=5, alleles_per_founder=9, length=500, snps_mean=7, seed=40 + k)
    j = write_json(lib, tmp_path / "lib.json")
    out = tmp_path / "lib.nb200idx"
    assert write_index(j, out, k)[0] == 0
    rc, inf, err = info(out, verify=1)
    assert rc == 0, err
    assert inf[0] == 1 and inf[1] == k
    assert inf[2:8] == host_stats(j, k)
    assert inf[8] % 256 == 0 and inf[8] >= 16 * inf[6]
    data = out.read_bytes()
    assert sections(data)[3][1] == inf[8] and struct.unpack_from("<Q", data, OFF_FILE_BYTES)[0] == len(data)


def test_verify_group_on_library(small_index):
    rc, inf, err = info(small_index, verify=1)
    assert rc == 0, err
    assert inf[2:4] == [12, 3] and inf[7] == 0


@pytest.mark.parametrize("lf", [None, "0.93"])
def test_verify_dense_transcripts_with_dual_entries(tmp_path, lf, monkeypatch):
    j = write_json(dense_dual_library(), tmp_path / "lib.json")
    for k in (8, 21, 32):
        out = tmp_path / ("lib%d.nb200idx" % k)
        if lf:
            monkeypatch.setenv("NB200_TABLE_LF", lf)
        assert write_index(j, out, k)[0] == 0
        monkeypatch.delenv("NB200_TABLE_LF", raising=False)      # NB200_TABLE_LF acts at build time only
        rc, inf, err = info(out, verify=1)
        assert rc == 0, err
        assert inf[1] == k and inf[2] == 450 and inf[2:8] == host_stats(j, k)[:4] + [inf[6], inf[7]]
        if lf:
            assert inf[6] < 3 * inf[4]                           # dense table: under 3 slots per k-mer (small tables get 8)


@pytest.mark.parametrize("section", [0, 1, 2])
def test_flipped_byte_in_host_section_is_refused(small_index, section):
    data = bytearray(small_index.read_bytes())
    off, n, _ = sections(data)[section]
    data[off + n // 2] ^= 0x10
    small_index.write_bytes(bytes(data))
    for verify in (0, 1):
        rc, _, err = info(small_index, verify)
        assert rc == _lib.EINVAL and "section %s fails its checksum" % SECTIONS[section] in err


def test_flipped_byte_in_image_is_refused_by_verify(small_index):
    data = bytearray(small_index.read_bytes())
    off, n, _ = sections(data)[3]
    data[off + 40] ^= 0x01                                       # inside the first bucket of the table
    small_index.write_bytes(bytes(data))
    assert info(small_index, verify=0)[0] == 0                   # the image is checked on request (and on every device load)
    rc, _, err = info(small_index, verify=1)
    assert rc == _lib.EINVAL and "device image fails its checksum" in err


def test_lookup_pass_catches_a_resealed_table(small_index):
    """A table whose checksums were recomputed after an edit: the lookup pass still finds the references that lost k-mers."""
    data = bytearray(small_index.read_bytes())
    off, n, _ = sections(data)[3]
    table = np.frombuffer(bytes(data[off:off + n]), "<u8").copy()
    keys = table[0::2][:64]
    used = np.nonzero(keys != np.uint64(0xFFFFFFFFFFFFFFFF))[0]
    assert len(used) > 4
    for e in used[:4]:
        table[2 * e + 1] ^= np.uint64(0x1)                      # class id of the entry: off by one
    data[off:off + 8 * len(table)] = table.tobytes()
    struct.pack_into("<Q", data, OFF_SECTIONS + 24 * 3 + 16, py_checksum(data[off:off + n]))
    reseal(data)
    small_index.write_bytes(bytes(data))
    rc, _, err = info(small_index, verify=1)
    assert rc == _lib.EINVAL and "do not find their reference" in err


def test_header_damage_truncation_magic_and_version(small_index):
    good = small_index.read_bytes()
    cases = []
    d = bytearray(good); d[OFF_N_KMERS] ^= 0x01; cases.append((d, "header fails its checksum"))
    cases.append((bytearray(good[:len(good) - 1000]), "is truncated"))
    cases.append((bytearray(good[:100]), "is truncated"))
    cases.append((bytearray(good + b"\0" * 8), "bytes after its end"))
    d = bytearray(good); d[:8] = b"NB200IDY"; cases.append((d, "bad magic"))
    d = bytearray(good); struct.pack_into("<I", d, OFF_VERSION, 99); cases.append((d, "has format version 99; this build reads version 1"))
    d = bytearray(good); struct.pack_into("<I", d, OFF_VERSION, 99); reseal(d); cases.append((d, "has format version 99"))
    for data, msg in cases:
        small_index.write_bytes(bytes(data))
        rc, _, err = info(small_index, verify=0)
        assert rc == _lib.EINVAL and msg in err, (msg, err)
    small_index.write_bytes(good)
    assert info(small_index)[0] == 0


def test_index_usage_errors(tmp_path, capsys, small_index):
    with pytest.raises(SystemExit) as e:
        main(["index", "--reference", "a.json,b.json", "--output", str(tmp_path / "x.nb200idx")])
    assert e.value.code == 2 and "one library per call" in capsys.readouterr().err
    with pytest.raises(SystemExit) as e:
        main(["index", "--reference", "a.json"])
    assert e.value.code == 2 and "--output" in capsys.readouterr().err
    lib, _ = synth.allele_family_library(n_founders=2, alleles_per_founder=3, length=200, seed=9)
    j = write_json(lib, tmp_path / "lib.json")
    out = tmp_path / "bad.nb200idx"
    for argv, msg in ([["-k", "33"], "k must be in 4..32"], [["-k", "3"], "k must be in 4..32"]):
        with pytest.raises(SystemExit) as e:
            main(["index", "--reference", str(j), "--output", str(out)] + argv)
        assert e.value.code == 1 and msg in capsys.readouterr().err
        assert not out.exists() and not os.path.exists(str(out) + ".tmp")
    assert frontend.index(str(tmp_path / "missing.json"), str(out)) == 1
    assert "cannot open library file" in capsys.readouterr().err
    assert frontend.index(str(small_index), str(out)) == 1
    assert "is an index file already" in capsys.readouterr().err
    rc, _ = write_index(j, tmp_path / "no" / "such" / "dir.nb200idx")
    assert rc == _lib.EIO
    with pytest.raises(_lib.NimbleB200Error, match="cannot open index file"):
        frontend.index_info(tmp_path / "missing.nb200idx")
    with pytest.raises(_lib.NimbleB200Error, match="bad magic"):
        frontend.index_info(j)
