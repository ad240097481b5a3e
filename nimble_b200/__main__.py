"""`python -m nimble_b200 <subcommand>` — same sub-commands and flags as `python -m nimble`
(nimble/__main__.py:373-468) for the hot path: generate, align, report.  `download` reports that
the aligner is built in; `fastq-to-bam` (nimble/__main__.py:424-431) runs its barcode correction on
the GPU; `fastq-to-counts` (an extension) runs fastq-to-bam and align --counts in one pass; `index` (an extension) saves a
library's k-mer index to a file that every command taking --reference loads without a build; `plot` is outside the hot
path (DESIGN.md §7)."""
import argparse
import sys

from . import __version__
from .frontend import align, align_10x, fastq_to_bam_with_barcodes, fastq_to_counts, generate, index, report


def main(argv=None):
    parser = argparse.ArgumentParser(description="nimble align (B200-native backend)")
    parser.add_argument("-v", "--version", action="version", version=f"nimble_b200 {__version__}")
    sub = parser.add_subparsers(title="subcommands", dest="subcommand")

    d = sub.add_parser("download")
    d.add_argument("--release", help="The release to download.", type=str, default=[])

    g = sub.add_parser("generate")
    g.add_argument("--file", help="The file to process.", type=str, required=True)
    g.add_argument("--opt-file", help="The optional file to process.", type=str, default=None)
    g.add_argument("--output_path", help="The path to the output file.", type=str, required=True)

    a = sub.add_parser("align")
    a.add_argument("--reference", help="The reference genome to align to.", type=str, required=True)
    a.add_argument("--output", help="The path to the output file (per-read TSV; optional with --counts).", type=str, default=None)
    a.add_argument("--input", help="The input reads.", type=str, required=True, nargs="+")
    a.add_argument("-c", "--num_cores", help="The number of cores to use for alignment.", type=int, default=1)
    a.add_argument("--strand_filter", help="Filter reads based on strand information.", type=str, default="unstranded")
    a.add_argument("--trim", help="<TARGET_LENGTH>:<STRICTNESS>, comma-separated, one entry per library", type=str, default="")
    a.add_argument("--tmpdir", help="Path to a temporary directory for sorting .bam files", type=str, default=None)
    a.add_argument("-k", "--kmer", help="k-mer length of the index (4..32; default: an index file's own, 20 for a JSON)", type=int, default=None)
    a.add_argument("--map", help="(extension) cell barcode whitelist: --input is a raw 10x R1/R2 FASTQ pair, fastq-to-bam runs in "
                                 "the same pass without writing a BAM", type=str, default=None)
    a.add_argument("--gpus", help="(extension) GPUs of this node to spread the reads over (default 1; also $NB200_GPUS)", type=int, default=None)
    a.add_argument("--cb-length", type=int, default=16)
    a.add_argument("--umi-length", type=int, default=12)
    a.add_argument("--counts", help="(extension) also write the counts TSV `report` would write, in the same pass (BAM with CB/UB tags); "
                                    "--output becomes optional", type=str, default=None)
    a.add_argument("--threshold", help="with --counts: proportional count threshold for filtering features (default: 0.05), as for report",
                   type=float, default=0.05)
    a.add_argument("--disable_thresholding", help="with --counts: disable the per-UMI proportional count thresholding algorithm",
                   action="store_true", default=False)
    a.add_argument("--correct-umis", help="(extension) with --counts: merge each UMI into a better-supported UMI of the same cell one "
                                          "substitution away before counting (DESIGN.md §2.12)", action="store_true", default=False)

    r = sub.add_parser("report")
    r.add_argument("-i", "--input", help="The input file.", type=str, required=True)
    r.add_argument("-o", "--output", help="The path to the output file.", type=str, required=True)
    r.add_argument("-s", "--summarize", help="CSV list of columns to summarize.", type=str, default=None)
    r.add_argument("-t", "--threshold", help="Proportional count threshold for filtering features (default: 0.05).",
                   type=float, default=0.05)
    r.add_argument("--disable_thresholding", help="Disable the per-UMI proportional count thresholding algorithm.",
                   action="store_true", default=False)
    r.add_argument("--correct-umis", help="(extension) merge each UMI into a better-supported UMI of the same cell one substitution "
                                          "away before counting (DESIGN.md §2.12)", action="store_true", default=False)

    f = sub.add_parser("fastq-to-bam")
    f.add_argument("--r1-fastq", help="Path to R1 FASTQ file.", type=str, required=True)
    f.add_argument("--r2-fastq", help="Path to R2 FASTQ file.", type=str, required=True)
    f.add_argument("--map", required=True, help="Cell barcode whitelist file (one CB per line, .gz or plain text)")
    f.add_argument("--output", help="Path for output BAM file.", type=str, required=True)
    f.add_argument("-c", "--num_cores", help="The number of cores to use for processing.", type=int, default=1)
    f.add_argument("--cb-length", help="Length of cell barcode (default: 16).", type=int, default=16)
    f.add_argument("--umi-length", help="Length of UMI (default: 12).", type=int, default=12)

    fc = sub.add_parser("fastq-to-counts", help="(extension) fastq-to-bam, then align --counts on its BAM, in one pass without the BAM")
    fc.add_argument("--reference", help="The reference library (comma-separated for several).", type=str, required=True)
    fc.add_argument("--r1-fastq", help="Path to R1 FASTQ file.", type=str, required=True)
    fc.add_argument("--r2-fastq", help="Path to R2 FASTQ file.", type=str, required=True)
    fc.add_argument("--map", required=True, help="Cell barcode whitelist file (one CB per line, .gz or plain text)")
    fc.add_argument("--counts", help="Path of the counts TSV (one per library, named as align names its outputs).", type=str, required=True)
    fc.add_argument("--output", help="Also write the per-read TSV align --map writes (one per library, named as align names its "
                                     "outputs), in the same pass", type=str, default=None)
    fc.add_argument("-c", "--num_cores", help="The number of host threads to use.", type=int, default=1)
    fc.add_argument("--strand_filter", help="Filter reads based on strand information.", type=str, default="unstranded")
    fc.add_argument("--trim", help="<TARGET_LENGTH>:<STRICTNESS>, comma-separated, one entry per library", type=str, default="")
    fc.add_argument("-k", "--kmer", help="k-mer length of the index (4..32; default: an index file's own, 20 for a JSON)", type=int, default=None)
    fc.add_argument("--gpus", help="GPUs of this node to spread the reads over (default 1; also $NB200_GPUS)", type=int, default=None)
    fc.add_argument("--cb-length", help="Length of cell barcode (default: 16).", type=int, default=16)
    fc.add_argument("--umi-length", help="Length of UMI (default: 12).", type=int, default=12)
    fc.add_argument("--threshold", help="Proportional count threshold for filtering features (default: 0.05), as for report",
                    type=float, default=0.05)
    fc.add_argument("--disable_thresholding", help="Disable the per-UMI proportional count thresholding algorithm.",
                    action="store_true", default=False)
    fc.add_argument("--correct-umis", help="(extension) merge each UMI into a better-supported UMI of the same cell one substitution "
                                           "away before counting (DESIGN.md §2.12)", action="store_true", default=False)

    ix = sub.add_parser("index", help="(extension) build one library's k-mer index on the host and save it; --reference LIB.nb200idx "
                                      "then loads it without a build")
    ix.add_argument("--reference", help="The reference library JSON (one per call).", type=str, required=True)
    ix.add_argument("--output", help="Path of the index file (e.g. LIB.nb200idx).", type=str, required=True)
    ix.add_argument("-k", "--kmer", help="k-mer length of the index (4..32, default: 20)", type=int, default=None)
    ix.add_argument("-c", "--num_cores", help="The number of host threads to use (default: all cores).", type=int, default=0)

    pl = sub.add_parser("plot")          # visualisation: outside the hot path (DESIGN.md §7); flags accepted so scripts fail clearly
    pl.add_argument("--input_file", "-i", type=str, required=False)
    pl.add_argument("--output_file", "-o", type=str, required=False)

    args = parser.parse_args(argv)
    if args.subcommand == "download":
        print("nimble_b200: the aligner is the in-tree CUDA library (libnimble_b200.so); nothing to download.")
    elif args.subcommand == "generate":
        generate(args.file, args.opt_file, args.output_path)
    elif args.subcommand == "align" and args.output is None and args.counts is None:
        parser.error("align needs --output, --counts or both")
    elif args.subcommand == "align" and args.correct_umis and args.counts is None:
        parser.error("--correct-umis needs --counts")
    elif args.subcommand == "align" and args.map:
        if args.counts is not None:
            parser.error("--counts does not combine with --map: run align --map, then report on its per-read TSV")
        if len(args.input) != 2:
            parser.error("--map needs exactly two --input files (R1 and R2 FASTQ)")
        if args.trim:
            print("nimble_b200: --trim is applied by the streaming file path only; ignored with --map "
                  "(run fastq-to-bam, then align --trim on its BAM)", file=sys.stderr)
        sys.exit(align_10x(args.reference, args.output, args.input[0], args.input[1], args.map, args.num_cores, args.strand_filter,
                           args.cb_length, args.umi_length, k=args.kmer, gpus=args.gpus))
    elif args.subcommand == "align":
        sys.exit(align(args.reference, args.output, args.input, args.num_cores, args.strand_filter, args.trim,
                       args.tmpdir, k=args.kmer, gpus=args.gpus, counts=args.counts, threshold=args.threshold,
                       disable_thresholding=args.disable_thresholding, correct_umis=args.correct_umis))
    elif args.subcommand == "report":
        cols = args.summarize.split(",") if args.summarize else None
        report(args.input, args.output, cols, args.threshold, args.disable_thresholding, correct_umis=args.correct_umis)
    elif args.subcommand == "plot":
        print("nimble_b200: `plot` (HTML report, nimble/report_generation.py) is not part of the B200 backend; the per-read TSV "
              "written by `align` carries every column it reads, so `python -m nimble plot` works on it unchanged.", file=sys.stderr)
        sys.exit(2)
    elif args.subcommand == "fastq-to-bam":
        fastq_to_bam_with_barcodes(args.r1_fastq, args.r2_fastq, args.map, args.output, args.num_cores,
                                   args.cb_length, args.umi_length)
    elif args.subcommand == "fastq-to-counts":
        sys.exit(fastq_to_counts(args.reference, args.r1_fastq, args.r2_fastq, args.map, args.counts, args.num_cores, args.strand_filter,
                                 args.trim, k=args.kmer, gpus=args.gpus, cb_length=args.cb_length, umi_length=args.umi_length,
                                 threshold=args.threshold, disable_thresholding=args.disable_thresholding,
                                 correct_umis=args.correct_umis, output=args.output))
    elif args.subcommand == "index":
        if "," in args.reference:
            parser.error("index takes one library per call")
        sys.exit(index(args.reference, args.output, k=args.kmer, num_cores=args.num_cores))
    else:
        parser.print_help()


if __name__ == "__main__":
    main()
