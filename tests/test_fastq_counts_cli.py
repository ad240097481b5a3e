"""Usage errors of `fastq-to-counts` (no GPU needed: they are refused before any device work)."""
import pytest

from nimble_b200.__main__ import main


def test_fastq_to_counts_needs_its_inputs(capsys):
    with pytest.raises(SystemExit) as e:
        main(["fastq-to-counts", "--reference", "lib.json", "--r1-fastq", "r1.fastq", "--r2-fastq", "r2.fastq", "--counts", "c.tsv"])
    assert e.value.code == 2 and "--map" in capsys.readouterr().err
    with pytest.raises(SystemExit) as e:
        main(["fastq-to-counts", "--reference", "lib.json", "--r1-fastq", "r1.fastq", "--r2-fastq", "r2.fastq", "--map", "wl.txt"])
    assert e.value.code == 2 and "--counts" in capsys.readouterr().err


def test_fastq_to_counts_bad_trim(capsys):
    with pytest.raises(SystemExit) as e:
        main(["fastq-to-counts", "--reference", "a.json,b.json", "--r1-fastq", "r1.fastq", "--r2-fastq", "r2.fastq", "--map", "wl.txt",
              "--counts", "c.tsv", "--trim", "70:0.6"])
    assert e.value.code == 1 and "one <TARGET_LENGTH>:<STRICTNESS> entry per library" in capsys.readouterr().err
