"""Usage errors of `align --counts` (no GPU needed: argparse refuses them before any work)."""
import pytest

from nimble_b200.__main__ import main


def test_align_needs_output_or_counts(capsys):
    with pytest.raises(SystemExit) as e:
        main(["align", "--reference", "lib.json", "--input", "in.bam"])
    assert e.value.code == 2 and "--output, --counts or both" in capsys.readouterr().err


def test_counts_does_not_combine_with_map(capsys):
    with pytest.raises(SystemExit) as e:
        main(["align", "--reference", "lib.json", "--input", "r1.fastq.gz", "r2.fastq.gz", "--map", "wl.txt", "--counts", "c.tsv"])
    assert e.value.code == 2 and "--counts does not combine with --map" in capsys.readouterr().err
    with pytest.raises(SystemExit) as e:
        main(["align", "--reference", "lib.json", "--output", "o.tsv", "--input", "r1.fastq.gz", "r2.fastq.gz", "--map", "wl.txt",
              "--counts", "c.tsv"])
    assert e.value.code == 2
