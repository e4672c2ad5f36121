"""TEST INFRASTRUCTURE ONLY: ctypes front-end of tests/tandem_report_oracle.c (the tandem-repeat report of `--reportTRF`,
DESIGN §2 R1-R6) and the oracle pipelines of the `_TRF.gff3` file of `mimeo filter` and `mimeo map`: runs from
oracle.tandem_oracle.mask, one row per run from tro_report, printed fields formatted here from the integers."""
from __future__ import annotations

import ctypes as C
import math
import os
import subprocess
from typing import Dict, Tuple

import numpy as np

from oracle import tandem_oracle as to

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, 'tandem_report_oracle.c')
SO = os.path.join(HERE, 'emu', '_build', 'libtandem_report_oracle.so')
HEADER = '##gff-version 3\n##seqid\tsource\ttype\tstart\tend\tscore\tstrand\tphase\tattributes\n'
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        if not os.path.exists(SO) or os.path.getmtime(SO) < os.path.getmtime(SRC):
            os.makedirs(os.path.dirname(SO), exist_ok=True)
            tmp = f'{SO}.{os.getpid()}.tmp'
            subprocess.check_call([os.environ.get('CC', 'gcc'), '-O2', '-Wall', '-Wextra', '-std=gnu11', '-shared', '-fPIC', '-o', tmp, SRC])
            os.replace(tmp, SO)
        l = C.CDLL(SO)
        l.tro_report.restype = C.c_int
        l.tro_report.argtypes = [C.c_void_p, C.c_long, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_char_p]
        _LIB = l
    return _LIB


def report(run, match=2, mismatch=7, maxperiod=50, **_ignored) -> Tuple[int, int, int, Tuple[int, int, int, int], str]:
    """(period, score, matches, (A, C, G, T counts), consensus) of one run (ASCII, length >= 2)."""
    u = to._ascii(run)
    out = np.zeros(7, np.int64)
    cons = C.create_string_buffer(max(1, maxperiod))
    if lib().tro_report(u.ctypes.data, len(u), match, mismatch, maxperiod, out.ctypes.data, cons) != 0:
        raise ValueError('tandem report oracle: bad arguments')
    p = int(out[0])
    return p, int(out[1]), int(out[2]), tuple(int(v) for v in out[3:7]), cons.raw[:p].decode()


def gff_row(seqid: str, start: int, end: int, number: int, rep, extra: str = '') -> str:
    """One `_TRF.gff3` row of a run of L = end - start + 1 bases."""
    p, score, matches, counts, cons = rep
    L = end - start + 1
    tot = sum(counts)
    ent = sum(c / tot * math.log2(tot / c) for c in counts if c) if tot else 0.0
    comp = ','.join(f'{b}:{100 * c // L}' for b, c in zip('ACGT', counts))
    return (f'{seqid}\tmimeo-trf\ttandem_repeat\t{start}\t{end}\t{score}\t+\t.\tID=TR_{number:05d};period={p};copies={L / p:.1f};'
            f'consensus={cons};pmatch={100 * matches // L};composition={comp};entropy={ent:.2f}{extra}\n')


def fasta_report(records, params: Dict[str, int] = None) -> str:
    """`mimeo filter --reportTRF`: every (id, sequence) record in input order, its runs ascending, record-local 1-based."""
    p = dict(to.DEFAULTS, **(params or {}))
    rows = []
    for rid, seq in records:
        for a, e in (to.mask(seq, **p)[1] if len(seq) else []):
            rows.append(gff_row(rid, a + 1, e + 1, len(rows) + 1, report(to._ascii(seq)[a:e + 1], **p)))
    return HEADER + ''.join(rows)


def map_report(gff_text: str, agenome: Dict[str, object], params: Dict[str, int] = None) -> str:
    """`mimeo map --maxtandem --reportTRF` on the GFF3 of the oracle pipeline (before the filter): every row in file order,
    the runs of its A-genome span [start1 - 1, end1) ascending, genome coordinates, `;hit=<ID>` appended."""
    p = dict(to.DEFAULTS, **(params or {}))
    rows = []
    for line in gff_text.splitlines():
        if line.startswith('#'):
            continue
        c = line.split('\t')
        uid = dict(kv.split('=', 1) for kv in c[8].split(';'))['ID']
        s1, L = int(c[3]), int(c[4]) - int(c[3]) + 1
        span = to._ascii(agenome[c[0]])[s1 - 1:s1 - 1 + L]
        for a, e in to.mask(span, **p)[1]:
            rows.append(gff_row(c[0], s1 + a, s1 + e, len(rows) + 1, report(span[a:e + 1], **p), f';hit={uid}'))
    return HEADER + ''.join(rows)


def fasta_text_report(text: str, params: Dict[str, int] = None) -> str:
    """fasta_report of a FASTA text, records parsed by tests/filter_reference.py (id = first word of the header)."""
    from tests import filter_reference as fr
    return fasta_report([((h.split() or [''])[0], s.encode()) for h, s in fr.fasta_records(text)], params)
