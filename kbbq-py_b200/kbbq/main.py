#!/usr/bin/env python3
"""CLI of the drop-in (reference: kbbq/main.py:26-89).  Only `recalibrate` is on the hot path;
`benchmark` and `plot` need BAM / VCF / matplotlib tooling and are out of scope (SURVEY.md section 8)."""
import argparse
import sys

import kbbq
from kbbq import recalibrate as re


def recalibrate(args):
    re.recalibrate(bam=args.bam, fastq=args.fastq, infer_rg=args.infer_rg,
                   use_oq=args.use_oq, set_oq=args.set_oq, gatkreport=args.gatkreport,
                   reads=args.reads, kmer_size=args.kmer_size, min_count=args.min_count, kmer_correct=args.correct)


def _int_in(lo, hi):
    def parse(text):
        v = int(text)
        if not lo <= v <= hi:
            raise argparse.ArgumentTypeError("%d is not in %d..%d" % (v, lo, hi))
        return v
    return parse


def _out_of_scope(name):
    def run(args):
        raise NotImplementedError("`kbbq %s` is outside the B200 hot path; use the reference for it" % name)
    return run


def main():
    parser = argparse.ArgumentParser(description='K-mer Based Base Quality score recalibration')
    parser.add_argument('-v', '--version', action='version', version=kbbq.__version__)
    subparsers = parser.add_subparsers(title='command', description="valid commands")
    helpfn = lambda args: parser.print_help()
    parser.set_defaults(command=helpfn)
    help_parser = subparsers.add_parser('help', description='Print help information')
    help_parser.set_defaults(command=helpfn)

    oq_help = 'Use the OQ tag to get quality scores when working with a BAM file. Does nothing if a fastq file is provided.'
    recalibrate_parser = subparsers.add_parser('recalibrate', description='Recalibrate a BAM or FASTQ file')
    recalibrate_input = recalibrate_parser.add_mutually_exclusive_group(required=True)
    recalibrate_input.add_argument('-b', '--bam', help='BAM to recalibrate')
    recalibrate_input.add_argument('-f', '--fastq', nargs=2,
                                   help='FASTQ file to recalibrate and a corrected version from your favorite error corrector.')
    recalibrate_input.add_argument('-r', '--reads',
                                   help='FASTQ file to recalibrate, its errors found on the GPU from its own k-mer counts.')
    recalibrate_parser.add_argument('-k', '--kmer-size', type=_int_in(1, 31), default=23,
                                    help='k-mer length of --reads (1..31, default 23).')
    recalibrate_parser.add_argument('--min-count', type=_int_in(0, 2 ** 31 - 1), default=0,
                                    help='Count from which a k-mer of --reads is trusted; 0 (default) takes the first '
                                         'valley of the count histogram.')
    recalibrate_parser.add_argument('--correct', action='store_true',
                                    help='with -r: find each error by correcting the read against its trusted k-mers')
    recalibrate_parser.add_argument('-u', '--use-oq', action='store_true', help=oq_help)
    recalibrate_parser.add_argument('-s', '--set-oq', action='store_true',
                                    help='Set the \'OQ\' flag prior to recalibration. Only works when producing BAM output.')
    recalibrate_parser.add_argument('-g', '--gatkreport',
                                    help='If the given path points to an existing GATK report, load the model from the '
                                         'report instead of calculating it. If the file doesn\'t exist, save the '
                                         'calculated model to the given path.')
    recalibrate_parser.add_argument('--infer-rg', action='store_true',
                                    help='Attempt to infer the read group from a FASTQ read. Only works with FASTQ input. '
                                         'The default behavior is to treat each input FASTQ file as its own read group.')
    recalibrate_parser.set_defaults(command=recalibrate)

    for name in ('benchmark', 'plot'):
        sub = subparsers.add_parser(name, description='(reference-only command, not part of the B200 hot path)')
        sub.add_argument('rest', nargs=argparse.REMAINDER)
        sub.set_defaults(command=_out_of_scope(name))

    args = parser.parse_args()
    if getattr(args, 'correct', False) and args.reads is None:
        recalibrate_parser.error('--correct needs -r/--reads')
    args.command(args)


if __name__ == '__main__':
    main()
