"""`mimeo filter`: drop the records of a FASTA library that are more than --maxtandem percent tandem repeat (the reference's
run_filter / trfFasta step, SURVEY 2.1 and 3.5: SSR filtering of repeat libraries, e.g. segments extracted from `mimeo x` or
`self` output). The reference's CLI is not in the tree; this one reuses `mimeo map`'s --t* options, and every record is masked
as a whole on the GPU under this project's own statement (DESIGN §2, T1-T4), not Tandem Repeats Finder: --TRFpath, --tPM and
--tPI are accepted and have no effect. --writeTRF also writes every record with its masked positions replaced by N to
`<outfile without .fa/.fasta/.fna>_TRFmasked.fa`."""
import argparse
import logging
import os
import sys

from . import tandem
from ._cli_common import add_loglevel, add_version
from .fasta import read_fasta
from .logs import init_logging


def mainArgs() -> argparse.Namespace:
    parser = argparse.ArgumentParser(description='Remove tandem-repeat-rich sequences from a FASTA library.', prog='mimeo-filter')
    add_version(parser)
    parser.add_argument('--infile', type=str, default=None, help='FASTA library to filter.')
    parser.add_argument('--outfile', type=str, default='mimeo_filtered.fa', help='Name of the filtered FASTA file.')
    parser.add_argument('-d', '--outdir', type=str, default=None, help='Write output files to this directory. (Default: cwd)')
    parser.add_argument('--TRFpath', type=str, default='trf', help='Accepted for compatibility; the tandem repeat mask runs on the GPU.')
    parser.add_argument('--tmatch', type=int, default=2, help='Tandem mask matching weight (>= 1)')
    parser.add_argument('--tmismatch', type=int, default=7, help='Tandem mask mismatch penalty (>= 0)')
    parser.add_argument('--tdelta', type=int, default=7, help='Tandem mask indel penalty (>= 0)')
    parser.add_argument('--tPM', type=int, default=80, help='Accepted for compatibility; no effect (DESIGN T1).')
    parser.add_argument('--tPI', type=int, default=10, help='Accepted for compatibility; no effect (DESIGN T1).')
    parser.add_argument('--tminscore', type=int, default=50, help='Tandem mask minimum alignment score (>= 1)')
    parser.add_argument('--tmaxperiod', type=int, default=50, help='Tandem mask maximum period (1..256)')
    parser.add_argument('--maxtandem', type=float, default=40.0,
                        help='Max percentage of a sequence which may be masked as tandem repeat (0..100; 0 drops any sequence with a masked base).')
    parser.add_argument('--writeTRF', action='store_true', default=False,
                        help='Also write every input sequence with its masked positions replaced by N.')
    add_loglevel(parser)
    return parser.parse_args()


def main() -> None:
    args = mainArgs()
    init_logging(loglevel=args.loglevel)
    logging.info('Starting tandem repeat filter.')
    tparams = tandem.params(args.tmatch, args.tmismatch, args.tdelta, args.tminscore, args.tmaxperiod)
    if not 0.0 <= args.maxtandem <= 100.0:
        raise ValueError('--maxtandem must be in 0..100')
    if not args.infile or not os.path.isfile(args.infile):
        logging.error('Input fasta not found: %s' % args.infile)
        sys.exit(1)
    records = read_fasta(args.infile)
    if not records:
        logging.error('No sequences found in %s' % args.infile)
        sys.exit(1)
    if args.outdir:
        outdir = os.path.abspath(args.outdir)
        if not os.path.isdir(outdir):
            logging.info('Create output directory: %s' % outdir)
            os.makedirs(outdir)
    else:
        outdir = os.getcwd()
    outfile = os.path.join(outdir, args.outfile)
    tandem.write_filtered_fasta(records, outfile, args.maxtandem, tparams, tandem.masked_fasta_path(outfile) if args.writeTRF else None)
    logging.info('Finished!')
