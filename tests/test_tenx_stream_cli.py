"""CLI wiring of the streaming 10x routes (no GPU needed: the front-end functions are replaced)."""
import pytest

import nimble_b200.__main__ as M
from nimble_b200.__main__ import main


def _capture(monkeypatch, name):
    seen = {}

    def fake(*args, **kw):
        seen["args"], seen["kw"] = args, kw
        return 0
    monkeypatch.setattr(M, name, fake)
    return seen


def test_fastq_to_counts_output_reaches_the_front_end(monkeypatch):
    seen = _capture(monkeypatch, "fastq_to_counts")
    with pytest.raises(SystemExit) as e:
        main(["fastq-to-counts", "--reference", "lib.json", "--r1-fastq", "r1.fastq", "--r2-fastq", "r2.fastq", "--map", "wl.txt",
              "--counts", "c.tsv", "--output", "per_read.tsv", "--gpus", "2"])
    assert e.value.code == 0 and seen["kw"]["output"] == "per_read.tsv" and seen["kw"]["gpus"] == 2
    with pytest.raises(SystemExit):
        main(["fastq-to-counts", "--reference", "lib.json", "--r1-fastq", "r1.fastq", "--r2-fastq", "r2.fastq", "--map", "wl.txt",
              "--counts", "c.tsv"])
    assert seen["kw"]["output"] is None


def test_align_map_passes_gpus(monkeypatch):
    seen = _capture(monkeypatch, "align_10x")
    with pytest.raises(SystemExit) as e:
        main(["align", "--reference", "lib.json", "--output", "o.tsv", "--input", "r1.fastq.gz", "r2.fastq.gz", "--map", "wl.txt",
              "--gpus", "2"])
    assert e.value.code == 0 and seen["kw"]["gpus"] == 2 and seen["args"][:5] == ("lib.json", "o.tsv", "r1.fastq.gz", "r2.fastq.gz", "wl.txt")


def test_counts_with_map_still_refused(monkeypatch, capsys):
    seen = _capture(monkeypatch, "align_10x")
    with pytest.raises(SystemExit) as e:
        main(["align", "--reference", "lib.json", "--input", "r1.fastq.gz", "r2.fastq.gz", "--map", "wl.txt", "--counts", "c.tsv",
              "--gpus", "2"])
    assert e.value.code == 2 and "--counts does not combine with --map" in capsys.readouterr().err and not seen
