"""The tandem-repeat filter of `mimeo map --maxtandem` (the reference's trfFilter step, SURVEY 3.3). The mask is this
project's own statement computed on the GPU (DESIGN §2, T1-T4; `mb2_tandem_mask`), not Tandem Repeats Finder."""
from __future__ import annotations

import ctypes as C
import logging
from typing import Dict, List, Sequence, Tuple

import numpy as np

from . import _lib
from .engine import TAB_HEADER

MAX_PERIOD = 256


def params(match=2, mismatch=7, delta=7, minscore=50, maxperiod=50) -> Dict[str, int]:
    """The mask parameters (--tmatch, --tmismatch, --tdelta, --tminscore, --tmaxperiod); ValueError when out of range."""
    p = dict(match=int(match), mismatch=int(mismatch), delta=int(delta), minscore=int(minscore), maxperiod=int(maxperiod))
    if p['match'] < 1:
        raise ValueError('--tmatch must be at least 1')
    if p['mismatch'] < 0 or p['delta'] < 0:
        raise ValueError('--tmismatch and --tdelta must be at least 0')
    if p['minscore'] < 1:
        raise ValueError('--tminscore must be at least 1')
    if not 1 <= p['maxperiod'] <= MAX_PERIOD:
        raise ValueError(f'--tmaxperiod must be in 1..{MAX_PERIOD}')
    if p['minscore'] + p['mismatch'] > 65535:
        raise ValueError('--tminscore + --tmismatch must be at most 65535')
    return p


def _cparams(p: Dict[str, int]) -> _lib.TandemParams:
    c = _lib.TandemParams()
    _lib.lib().mb2_default_tandem_params(C.byref(c))
    for k, v in p.items():
        setattr(c, k, int(v))
    return c


def _spans(scaf, start0, length):
    return (np.ascontiguousarray(scaf, dtype=np.int32), np.ascontiguousarray(start0, dtype=np.int64),
            np.ascontiguousarray(length, dtype=np.int64))


def masked_counts(genome, scaf, start0, length, p: Dict[str, int]) -> np.ndarray:
    """Masked positions of every span (scaffold index, 0-based start, length). `genome` is a device Genome or a sequence of
    ASCII scaffolds (uploaded for the call)."""
    from .genome import Genome
    g = genome if isinstance(genome, Genome) else Genome([str(k) for k in range(len(genome))], genome)
    try:
        s, b, n = _spans(scaf, start0, length)
        out = np.zeros(len(s), dtype=np.uint64)
        _lib.check(_lib.lib().mb2_tandem_mask(g.handle, s.ctypes.data, b.ctypes.data, n.ctypes.data, len(s), C.byref(_cparams(p)),
                                              out.ctypes.data))
        return out
    finally:
        if g is not genome:
            g.close()


def masked_runs(genome, scaf, start0, length, p: Dict[str, int], store_budget: int = 0) -> Tuple[np.ndarray, List[List[Tuple[int, int]]]]:
    """Test hook: (masked counts, merged masked runs of every span as span-local closed (start, end) pairs)."""
    s, b, n = _spans(scaf, start0, length)
    out = np.zeros(len(s), dtype=np.uint64)
    r = _lib.TandemRuns()
    _lib.check(_lib.lib().mb2_test_tandem_mask(genome.handle, s.ctypes.data, b.ctypes.data, n.ctypes.data, len(s), C.byref(_cparams(p)),
                                               int(store_budget), out.ctypes.data, C.byref(r)))
    try:
        off = np.ctypeslib.as_array(r.off, shape=(len(s) + 1,)).copy()
        tot = int(off[-1])
        st = np.ctypeslib.as_array(r.start, shape=(max(tot, 1),))[:tot].tolist()
        en = np.ctypeslib.as_array(r.end, shape=(max(tot, 1),))[:tot].tolist()
    finally:
        _lib.lib().mb2_free_tandem_runs(C.byref(r))
    return out, [list(zip(st[off[k]:off[k + 1]], en[off[k]:off[k + 1]])) for k in range(len(s))]


def _tab_key(fields: Sequence[str]) -> Tuple[str, ...]:
    return tuple(fields[:10])


def _gff_key(cols: Sequence[str]) -> Tuple[str, ...]:
    """The 10 .tab fields a `mimeo map` GFF3 row was formatted from (B_locus = name2_strand2_start2_end2)."""
    attrs = dict(a.split('=', 1) for a in cols[8].rstrip('\n').split(';'))
    name2, strand2, start2, end2 = attrs['B_locus'].rsplit('_', 3)
    return (cols[0], cols[6], cols[3], cols[4], name2, strand2, start2, end2, cols[5], attrs['identity'])


def filter_map_rows(rows: List[str], adir: str, maxtandem: float, p: Dict[str, int]) -> List[bool]:
    """For each GFF3 feature row of `mimeo map`: keep it unless more than maxtandem percent of its A-genome span
    [start1 - 1, end1) is masked."""
    from .fasta import dir_records
    names, seqs = [], []
    for rid, _h, seq, _p in dir_records(adir):
        names.append(rid)
        seqs.append(seq)
    index = {n: k for k, n in enumerate(names)}
    cols = [r.split('\t') for r in rows]
    missing = sorted({c[0] for c in cols if c[0] not in index})
    if missing:
        raise RuntimeError(f'A-genome scaffold {missing[0]!r} of an alignment is not in {adir}')
    scaf = np.array([index[c[0]] for c in cols], dtype=np.int32)
    s1 = np.array([int(c[3]) for c in cols], dtype=np.int64)
    e1 = np.array([int(c[4]) for c in cols], dtype=np.int64)
    length = e1 - s1 + 1
    if (s1 < 1).any() or (length < 1).any():
        raise RuntimeError('malformed alignment span: need 1 <= start1 <= end1')
    m = masked_counts(seqs, scaf, s1 - 1, length, p) if len(rows) else np.zeros(0, np.uint64)
    return [not (100.0 * float(mm) / float(L) > maxtandem) for mm, L in zip(m.tolist(), length.tolist())]


def write_filtered_map(infile: str, body: str, gffout: str, chrlens, adir: str, maxtandem: float, p: Dict[str, int],
                       trf_out: str = None) -> int:
    """`mimeo map` with the tandem filter: the GFF3 feature rows (UIDs already assigned in import_Align order) of the hits
    that pass, under the unchanged headers; with trf_out also TAB_HEADER + the .tab lines of those hits, byte for byte, in
    GFF order. Returns the number of rows kept."""
    rows = body.splitlines(keepends=True)
    keep = filter_map_rows(rows, adir, maxtandem, p)
    kept = [r for r, k in zip(rows, keep) if k]
    logging.info('Tandem repeat filter: %d of %d alignments kept (maxtandem %s%%)', len(kept), len(rows), maxtandem)
    if not kept:
        logging.warning('Every alignment was removed by the tandem repeat filter; writing headers only.')
    if gffout:
        with open(gffout, 'w', encoding='utf-8', errors='surrogateescape') as f:
            f.write('##gff-version 3\n')
            for name, maxlen in (chrlens or []):
                f.write(f'##sequence-region {name} 1 {maxlen}\n')
            f.write('##seqid\tsource\ttype\tstart\tend\tscore\tstrand\tphase\tattributes\n')
            f.write(''.join(kept))
    if trf_out:
        lines: Dict[Tuple[str, ...], List[str]] = {}
        with open(infile, encoding='utf-8', errors='surrogateescape', newline='') as f:
            for raw in f:
                li = raw.strip()
                if not li or li.startswith('#'):
                    continue
                lines.setdefault(_tab_key(li.split()), []).append(raw if raw.endswith('\n') else raw + '\n')
        with open(trf_out, 'w', encoding='utf-8', errors='surrogateescape', newline='') as f:
            f.write(TAB_HEADER)
            for r, k in zip(rows, keep):
                line = lines[_gff_key(r.split('\t'))].pop(0)    # equal rows keep file order (the sort is stable)
                if k:
                    f.write(line)
    return len(kept)


def trf_path(outtab: str) -> str:
    """`<outfile without .tab>_TRFfiltered.tab`."""
    stem = outtab[:-4] if outtab.endswith('.tab') else outtab
    return stem + '_TRFfiltered.tab'
