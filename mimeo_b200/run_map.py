"""`mimeo map` (host mirror of src/mimeo/run_map.py). With --maxtandem, hits whose A-genome span is masked by more than
that percentage are dropped after numbering (import_Align -> tandem filter -> GFF3, SURVEY 3.3), so the surviving rows
keep their IDs. The mask is this project's own GPU statement (DESIGN §2, T1-T4), not Tandem Repeats Finder: --TRFpath,
--tPM and --tPI are accepted and have no effect. --writeTRF (with --maxtandem) also writes the .tab lines of the surviving
hits to `<outfile without .tab>_TRFfiltered.tab`. The same mask filters whole FASTA records in `mimeo filter` (run_filter.py)."""
import argparse
import logging
import os
import shutil
import sys
from typing import List

from . import tandem
from ._cli_common import add_loglevel, add_version
from .logs import init_logging
from .utils import chromlens, get_all_pairs, run_cmd, set_paths
from .wrappers import import_Align, map_LZ_cmds, map_gff_text, write_map_gff, writeGFFlines  # noqa: F401  (the pandas pair stays importable)


def mainArgs() -> argparse.Namespace:
    parser = argparse.ArgumentParser(description='Find all high-identity segments shared between genomes.', prog='mimeo-map')
    add_version(parser)
    parser.add_argument('--adir', type=str, default=None, help='Name of directory containing sequences from A genome.')
    parser.add_argument('--bdir', type=str, default=None, help='Name of directory containing sequences from B genome.')
    parser.add_argument('--afasta', type=str, default=None, help='A genome as multifasta.')
    parser.add_argument('--bfasta', type=str, default=None, help='B genome as multifasta.')
    parser.add_argument('-r', '--recycle', action='store_true', help='Use existing alignment "--outfile" if found.')
    parser.add_argument('-d', '--outdir', type=str, default=None, help='Write output files to this directory. (Default: cwd)')
    parser.add_argument('--gffout', type=str, default=None, help='Name of GFF3 annotation file. If not set, suppress output.')
    parser.add_argument('--outfile', type=str, default='mimeo_alignment.tab', help='Name of alignment result file.')
    parser.add_argument('--verbose', action='store_true', default=False, help='If set report alignment stage counters.')
    parser.add_argument('--label', type=str, default='BHit', help='Set annotation TYPE field in gff.')
    parser.add_argument('--prefix', type=str, default='BHit', help='ID prefix for B-genome hits annotated in A-genome.')
    parser.add_argument('--keeptemp', action='store_true', default=False, help='If set do not remove temp files.')
    parser.add_argument('--lzpath', type=str, default='lastz', help='Accepted for compatibility; alignment runs on the GPU.')
    parser.add_argument('--minIdt', type=int, default=60, help='Minimum alignment identity to report.')
    parser.add_argument('--minLen', type=int, default=100, help='Minimum alignment length to report.')
    parser.add_argument('--hspthresh', type=int, default=3000, help='Set HSP min score threshold.')
    parser.add_argument('--TRFpath', type=str, default='trf', help='Accepted for compatibility; the tandem repeat mask runs on the GPU.')
    parser.add_argument('--tmatch', type=int, default=2, help='Tandem mask matching weight (>= 1)')
    parser.add_argument('--tmismatch', type=int, default=7, help='Tandem mask mismatch penalty (>= 0)')
    parser.add_argument('--tdelta', type=int, default=7, help='Tandem mask indel penalty (>= 0)')
    parser.add_argument('--tPM', type=int, default=80, help='Accepted for compatibility; no effect (DESIGN T1).')
    parser.add_argument('--tPI', type=int, default=10, help='Accepted for compatibility; no effect (DESIGN T1).')
    parser.add_argument('--tminscore', type=int, default=50, help='Tandem mask minimum alignment score (>= 1)')
    parser.add_argument('--tmaxperiod', type=int, default=50, help='Tandem mask maximum period (1..256)')
    parser.add_argument('--maxtandem', type=float, default=None, help='Max percentage of an A-genome alignment which may be masked as tandem repeat.')
    parser.add_argument('--writeTRF', action='store_true', default=False, help='With --maxtandem, also write the alignments that pass the filter.')
    add_loglevel(parser)
    return parser.parse_args()


def main() -> None:
    args = mainArgs()
    init_logging(loglevel=args.loglevel)
    logging.info('Starting genome mapping workflow.')
    tparams = None
    if args.maxtandem:
        tparams = tandem.params(args.tmatch, args.tmismatch, args.tdelta, args.tminscore, args.tmaxperiod)
    adir_path, bdir_path, outdir, outtab, gffout, tempdir = set_paths(
        adir=args.adir, bdir=args.bdir, afasta=args.afasta, bfasta=args.bfasta, outdir=args.outdir, outtab=args.outfile,
        gffout=args.gffout, runtrf=args.maxtandem)
    pairs = get_all_pairs(Adir=adir_path, Bdir=bdir_path)
    logging.info('Number of pairs to align: %d', len(pairs))
    chrLens = chromlens(seqDir=adir_path)
    if not args.recycle or not os.path.isfile(outtab):
        if not pairs:
            logging.error('No files to align. Check --adir and --bdir contain at least one fasta each.')
            sys.exit(1)
        cmds: List[str] = map_LZ_cmds(lzpath=args.lzpath, pairs=pairs, minIdt=args.minIdt, minLen=args.minLen,
                                      hspthresh=args.hspthresh, outfile=outtab, verbose=args.verbose)
        logging.info('Running alignments...')
        run_cmd(cmds, verbose=args.verbose, keeptemp=args.keeptemp)
    # import_Align + writeGFFlines (still importable from .wrappers) in one native pass over the .tab file
    if tparams is None:
        write_map_gff(infile=outtab, gffout=gffout, chrlens=chrLens, prefix=args.prefix, minLen=args.minLen, minIdt=args.minIdt,
                      ftype=args.label)
    else:
        n, body = map_gff_text(outtab, args.prefix, args.minLen, args.minIdt, args.label)
        if n == 0:
            logging.warning('No alignments found in %s' % outtab)
            sys.exit(1)
        tandem.write_filtered_map(outtab, body, gffout, chrLens, adir_path, args.maxtandem, tparams,
                                  tandem.trf_path(outtab) if args.writeTRF else None)
    if tempdir and os.path.isdir(tempdir) and not args.keeptemp:
        shutil.rmtree(tempdir)
    logging.info('Finished!')
