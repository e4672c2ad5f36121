"""The tandem-repeat filters: `mimeo map --maxtandem` (the reference's trfFilter step, SURVEY 3.3) and `mimeo filter` (its
trfFasta step, SURVEY 3.5). The mask is this project's own statement computed on the GPU (DESIGN §2, T1-T4;
`mb2_tandem_mask`), not Tandem Repeats Finder. `--reportTRF` adds a GFF3 report of every masked run (period, copies,
consensus, purity, composition; DESIGN §2, R1-R6; `mb2_tandem_report`)."""
from __future__ import annotations

import ctypes as C
import logging
import math
from typing import Dict, List, NamedTuple, Optional, Sequence, Tuple

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


def _with_runs(nspans: int, call) -> Tuple[np.ndarray, List[List[Tuple[int, int]]]]:
    """Runs call(masked, runs) on an mb2_tandem_runs result and returns (masked counts, runs of every span as lists of
    span-local closed (start, end) pairs); the library's arrays are freed whatever happens."""
    out = np.zeros(nspans, dtype=np.uint64)
    r = _lib.TandemRuns()
    try:
        _lib.check(call(out.ctypes.data, C.byref(r)))
        off = np.ctypeslib.as_array(r.off, shape=(nspans + 1,)).copy()
        tot = int(off[-1])
        st = np.ctypeslib.as_array(r.start, shape=(max(tot, 1),))[:tot].tolist()
        en = np.ctypeslib.as_array(r.end, shape=(max(tot, 1),))[:tot].tolist()
    finally:
        _lib.lib().mb2_free_tandem_runs(C.byref(r))
    return out, [list(zip(st[off[k]:off[k + 1]], en[off[k]:off[k + 1]])) for k in range(nspans)]


def masked_runs(genome, scaf, start0, length, p: Dict[str, int], store_budget: int = 0) -> Tuple[np.ndarray, List[List[Tuple[int, int]]]]:
    """Test hook: (masked counts, merged masked runs of every span as span-local closed (start, end) pairs)."""
    s, b, n = _spans(scaf, start0, length)
    return _with_runs(len(s), lambda m, r: _lib.lib().mb2_test_tandem_mask(genome.handle, s.ctypes.data, b.ctypes.data, n.ctypes.data,
                                                                            len(s), C.byref(_cparams(p)), int(store_budget), m, r))


def record_masks(seqs: Sequence[np.ndarray], p: Dict[str, int], runs: bool = False) -> Tuple[np.ndarray, Optional[List[List[Tuple[int, int]]]]]:
    """`mimeo filter`: the masked positions of every record, each masked as one span [0, L), and with runs=True also its
    merged masked runs (closed (start, end) pairs; None otherwise). The records with L >= 1 go to the device as one Genome;
    a record with L = 0 never does (m = 0, no runs)."""
    from .genome import Genome
    lens = np.array([len(s) for s in seqs], dtype=np.int64)
    idx = np.flatnonzero(lens > 0)
    m = np.zeros(len(seqs), dtype=np.uint64)
    iv: Optional[List[List[Tuple[int, int]]]] = [[] for _ in seqs] if runs else None
    if not len(idx):
        return m, iv
    g = Genome([str(k) for k in idx.tolist()], [seqs[k] for k in idx.tolist()])
    try:
        s, b, n = _spans(np.arange(len(idx)), np.zeros(len(idx)), lens[idx])
        if runs:
            got, got_iv = _with_runs(len(s), lambda mm, r: _lib.lib().mb2_tandem_mask_runs(g.handle, s.ctypes.data, b.ctypes.data, n.ctypes.data,
                                                                                          len(s), C.byref(_cparams(p)), mm, r))
            for k, v in zip(idx.tolist(), got_iv):
                iv[k] = v
        else:
            got = masked_counts(g, s, b, n, p)
    finally:
        g.close()
    m[idx] = got
    return m, iv


class Repeat(NamedTuple):
    """The report of one masked run [start, end] (closed, span-local): R2 period, R6 score, R4 matches, R5 counts of A, C, G,
    T and the R3 consensus."""
    start: int
    end: int
    period: int
    score: int
    matches: int
    counts: Tuple[int, int, int, int]
    consensus: str


def _with_report(nspans: int, call) -> Tuple[np.ndarray, List[List[Repeat]]]:
    """Runs call(masked, runs, rep) on mb2_tandem_runs and mb2_tandem_repeats results and returns (masked counts, the
    Repeats of every span); the library's arrays are freed whatever happens."""
    out = np.zeros(nspans, dtype=np.uint64)
    r, rep = _lib.TandemRuns(), _lib.TandemRepeats()
    try:
        _lib.check(call(out.ctypes.data, C.byref(r), C.byref(rep)))
        off = np.ctypeslib.as_array(r.off, shape=(nspans + 1,)).tolist()
        tot = off[-1]

        def arr(ptr, n):
            return np.ctypeslib.as_array(ptr, shape=(max(n, 1),))[:n].tolist()
        st, en = arr(r.start, tot), arr(r.end, tot)
        per, score, mt, cnt = arr(rep.period, tot), arr(rep.score, tot), arr(rep.matches, tot), arr(rep.count, 4 * tot)
        coff = arr(rep.cons_off, tot + 1)
        cons = C.string_at(rep.consensus, coff[-1]).decode('ascii') if tot else ''
    finally:
        _lib.lib().mb2_free_tandem_runs(C.byref(r))
        _lib.lib().mb2_free_tandem_report(C.byref(rep))
    reps = [Repeat(st[x], en[x], per[x], score[x], mt[x], tuple(cnt[4 * x:4 * x + 4]), cons[coff[x]:coff[x + 1]]) for x in range(tot)]
    return out, [reps[off[k]:off[k + 1]] for k in range(nspans)]


def masked_reports(genome, scaf, start0, length, p: Dict[str, int]) -> Tuple[np.ndarray, List[List[Repeat]]]:
    """masked_counts and, from the same device call, the Repeat of every merged masked run of every span (runs ascending)."""
    from .genome import Genome
    g = genome if isinstance(genome, Genome) else Genome([str(k) for k in range(len(genome))], genome)
    try:
        s, b, n = _spans(scaf, start0, length)
        return _with_report(len(s), lambda m, r, rep: _lib.lib().mb2_tandem_report(g.handle, s.ctypes.data, b.ctypes.data, n.ctypes.data,
                                                                                     len(s), C.byref(_cparams(p)), m, r, rep))
    finally:
        if g is not genome:
            g.close()


def record_reports(seqs: Sequence[np.ndarray], p: Dict[str, int]) -> Tuple[np.ndarray, List[List[Repeat]]]:
    """`mimeo filter --reportTRF`: record_masks with the Repeat of every run of every record (record-local runs)."""
    lens = np.array([len(s) for s in seqs], dtype=np.int64)
    idx = np.flatnonzero(lens > 0)
    m = np.zeros(len(seqs), dtype=np.uint64)
    reps: List[List[Repeat]] = [[] for _ in seqs]
    if not len(idx):
        return m, reps
    got, got_reps = masked_reports([seqs[k] for k in idx.tolist()], np.arange(len(idx)), np.zeros(len(idx)), lens[idx], p)
    m[idx] = got
    for k, v in zip(idx.tolist(), got_reps):
        reps[k] = v
    return m, reps


REPORT_HEADER = '##gff-version 3\n##seqid\tsource\ttype\tstart\tend\tscore\tstrand\tphase\tattributes\n'


def report_row(seqid: str, start: int, end: int, number: int, r: Repeat, extra: str = '') -> str:
    """The `_TRF.gff3` row of run r printed at [start, end] (1-based, closed) as TR_<number>; extra is appended to the
    attributes. copies = L / period, pmatch = floor(100 matches / L), composition = floor(100 count / L), entropy in bits of
    the A/C/G/T composition."""
    L = r.end - r.start + 1
    tot = sum(r.counts)
    ent = sum(c / tot * math.log2(tot / c) for c in r.counts if c) if tot else 0.0
    comp = ','.join(f'{b}:{100 * c // L}' for b, c in zip('ACGT', r.counts))
    return (f'{seqid}\tmimeo-trf\ttandem_repeat\t{start}\t{end}\t{r.score}\t+\t.\tID=TR_{number:05d};period={r.period};'
            f'copies={L / r.period:.1f};consensus={r.consensus};pmatch={100 * r.matches // L};composition={comp};entropy={ent:.2f}{extra}\n')


def _tab_key(fields: Sequence[str]) -> Tuple[str, ...]:
    return tuple(fields[:10])


def _gff_key(cols: Sequence[str]) -> Tuple[str, ...]:
    """The 10 .tab fields a `mimeo map` GFF3 row was formatted from (B_locus = name2_strand2_start2_end2)."""
    attrs = dict(a.split('=', 1) for a in cols[8].rstrip('\n').split(';'))
    name2, strand2, start2, end2 = attrs['B_locus'].rsplit('_', 3)
    return (cols[0], cols[6], cols[3], cols[4], name2, strand2, start2, end2, cols[5], attrs['identity'])


def _map_spans(rows: List[str], adir: str):
    """(A-genome scaffolds, scaffold index, start1, length) of the A-genome span [start1 - 1, end1) of every GFF3 row."""
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
    return seqs, scaf, s1, length


def _keep(m: np.ndarray, length: np.ndarray, maxtandem: float) -> List[bool]:
    return [not (100.0 * float(mm) / float(L) > maxtandem) for mm, L in zip(m.tolist(), length.tolist())]


def filter_map_rows(rows: List[str], adir: str, maxtandem: float, p: Dict[str, int]) -> List[bool]:
    """For each GFF3 feature row of `mimeo map`: keep it unless more than maxtandem percent of its A-genome span
    [start1 - 1, end1) is masked."""
    seqs, scaf, s1, length = _map_spans(rows, adir)
    m = masked_counts(seqs, scaf, s1 - 1, length, p) if len(rows) else np.zeros(0, np.uint64)
    return _keep(m, length, maxtandem)


def report_map_rows(rows: List[str], adir: str, maxtandem: float, p: Dict[str, int]) -> Tuple[List[bool], str]:
    """filter_map_rows and, from the same device call, the `_TRF.gff3` text: every row's runs in row order, runs ascending,
    at genome coordinates start1 + a .. start1 + e, with `;hit=<ID of the row>`."""
    seqs, scaf, s1, length = _map_spans(rows, adir)
    m, reps = masked_reports(seqs, scaf, s1 - 1, length, p) if len(rows) else (np.zeros(0, np.uint64), [])
    out = []
    for row, a0, rr in zip(rows, s1.tolist(), reps):
        cols = row.split('\t')
        uid = dict(kv.split('=', 1) for kv in cols[8].rstrip('\n').split(';'))['ID']
        for r in rr:
            out.append(report_row(cols[0], a0 + r.start, a0 + r.end, len(out) + 1, r, f';hit={uid}'))
    return _keep(m, length, maxtandem), REPORT_HEADER + ''.join(out)


def write_filtered_map(infile: str, body: str, gffout: str, chrlens, adir: str, maxtandem: float, p: Dict[str, int],
                       trf_out: str = None, report_out: str = None) -> int:
    """`mimeo map` with the tandem filter: the GFF3 feature rows (UIDs already assigned in import_Align order) of the hits
    that pass, under the unchanged headers; with trf_out also TAB_HEADER + the .tab lines of those hits, byte for byte, in
    GFF order; with report_out also the `_TRF.gff3` report of every hit evaluated. Returns the number of rows kept."""
    rows = body.splitlines(keepends=True)
    if report_out is None:
        keep = filter_map_rows(rows, adir, maxtandem, p)
    else:
        keep, report = report_map_rows(rows, adir, maxtandem, p)
        with open(report_out, 'w', encoding='utf-8', errors='surrogateescape') as f:
            f.write(report)
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


def _tab_stem(outtab: str) -> str:
    return outtab[:-4] if outtab.endswith('.tab') else outtab


def trf_path(outtab: str) -> str:
    """`<outfile without .tab>_TRFfiltered.tab`."""
    return _tab_stem(outtab) + '_TRFfiltered.tab'


def map_report_path(outtab: str) -> str:
    """`<outfile without .tab>_TRF.gff3`."""
    return _tab_stem(outtab) + '_TRF.gff3'


def write_filtered_fasta(records: Sequence[Tuple[str, str, np.ndarray]], outfile: str, maxtandem: float, p: Dict[str, int],
                         masked_out: str = None, report_out: str = None) -> int:
    """`mimeo filter`: of the (id, header, seq) records, write to outfile, in input order, every record unless more than
    maxtandem percent of it is masked (a record with L = 0 is kept); with masked_out also write every record there with its
    masked positions replaced by N. Both files in SeqIO.write's layout. With report_out also write the `_TRF.gff3` report of
    every record's runs, in input order, at record-local 1-based coordinates. Returns the number of records kept."""
    from .fasta import write_fasta_record
    seqs = [r[2] for r in records]
    if report_out is None:
        m, runs = record_masks(seqs, p, runs=masked_out is not None)
    else:
        m, reps = record_reports(seqs, p)
        runs = [[(r.start, r.end) for r in rr] for rr in reps]
        rows = [(rid, r) for (rid, _h, _s), rr in zip(records, reps) for r in rr]
        with open(report_out, 'w', encoding='utf-8', errors='surrogateescape') as f:
            f.write(REPORT_HEADER + ''.join(report_row(rid, r.start + 1, r.end + 1, k + 1, r) for k, (rid, r) in enumerate(rows)))
    keep = [len(s) == 0 or not (100.0 * float(mm) / len(s) > maxtandem) for s, mm in zip(seqs, m.tolist())]
    with open(outfile, 'wb') as f:
        for (_rid, header, seq), k in zip(records, keep):
            if k:
                write_fasta_record(f, header, seq)
    if masked_out is not None:
        with open(masked_out, 'wb') as f:
            for (_rid, header, seq), iv in zip(records, runs):
                if iv:
                    seq = seq.copy()
                    for a, e in iv:
                        seq[a:e + 1] = ord('N')
                write_fasta_record(f, header, seq)
    kept = sum(keep)
    logging.info('Tandem repeat filter: %d of %d records kept (maxtandem %s%%)', kept, len(records), maxtandem)
    if not kept:
        logging.warning('Every record was removed by the tandem repeat filter; %s is empty.', outfile)
    return kept


def _fasta_stem(outfile: str) -> str:
    for ext in ('.fa', '.fasta', '.fna'):
        if outfile.endswith(ext):
            return outfile[:-len(ext)]
    return outfile


def masked_fasta_path(outfile: str) -> str:
    """`<outfile without .fa/.fasta/.fna>_TRFmasked.fa`."""
    return _fasta_stem(outfile) + '_TRFmasked.fa'


def fasta_report_path(outfile: str) -> str:
    """`<outfile without .fa/.fasta/.fna>_TRF.gff3`."""
    return _fasta_stem(outfile) + '_TRF.gff3'
