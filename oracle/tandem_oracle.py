"""
tandem_oracle.py -- TEST INFRASTRUCTURE ONLY: ctypes front-end of oracle/tandem_oracle.c (the tandem-repeat mask of
`mimeo map --maxtandem`, DESIGN §2 T1-T4) and the oracle statement of the filter that `mimeo map` applies with it:
drop the GFF rows whose A-genome span is masked above --maxtandem percent, and write the surviving .tab lines in GFF
order for --writeTRF. This is our own mask, not Tandem Repeats Finder.

Only tests/ and scripts/ may import this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Dict, List, Sequence, Tuple

import numpy as np

from . import annot_oracle as ao

HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

DEFAULTS = dict(match=2, mismatch=7, delta=7, minscore=50, maxperiod=50)


def lib():
    global _LIB
    if _LIB is None:
        so = os.path.join(HERE, '_build', 'libtandem_oracle.so')
        src = os.path.join(HERE, 'tandem_oracle.c')
        if not os.path.exists(so) or os.path.getmtime(so) < os.path.getmtime(src):
            # built here rather than by oracle/Makefile, with the same compiler flags; written under a temporary name
            # and renamed, so that a reader never loads a half-written library
            os.makedirs(os.path.dirname(so), exist_ok=True)
            tmp = f'{so}.{os.getpid()}.tmp'
            subprocess.check_call([os.environ.get('CC', 'gcc'), '-O3', '-march=native', '-Wall', '-Wextra', '-std=gnu11', '-shared',
                                   '-fPIC', '-o', tmp, src])
            os.replace(tmp, so)
        l = C.CDLL(so)
        l.tro_mask.restype = C.c_long
        l.tro_mask.argtypes = [C.c_void_p, C.c_long, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_long,
                               C.POINTER(C.c_long)]
        _LIB = l
    return _LIB


def _ascii(seq) -> np.ndarray:
    if isinstance(seq, str):
        seq = seq.encode()
    if isinstance(seq, (bytes, bytearray)):
        return np.frombuffer(bytes(seq), dtype=np.uint8)
    return np.ascontiguousarray(seq, dtype=np.uint8)


def mask(seq, match=2, mismatch=7, delta=7, minscore=50, maxperiod=50) -> Tuple[int, List[Tuple[int, int]]]:
    """(masked positions m, merged masked intervals [(start, end)] closed and 0-based) of one ASCII sequence."""
    s = _ascii(seq)
    cap = len(s) // 2 + 2
    st, en = np.zeros(cap, np.int64), np.zeros(cap, np.int64)
    k = C.c_long(0)
    m = lib().tro_mask(s.ctypes.data, len(s), match, mismatch, delta, minscore, maxperiod, st.ctypes.data, en.ctypes.data, cap,
                       C.byref(k))
    if m < 0:
        raise ValueError('tandem oracle: bad arguments')
    return int(m), list(zip(st[:k.value].tolist(), en[:k.value].tolist()))


def masked_counts(seqs: Sequence, scaf, start0, length, params: Dict[str, int] = None) -> np.ndarray:
    """m of every span (scaffold index into seqs, 0-based start, length): the oracle twin of mimeo_b200.tandem.masked_counts."""
    p = dict(DEFAULTS, **(params or {}))
    out = np.zeros(len(scaf), dtype=np.uint64)
    for k, (c, s, n) in enumerate(zip(np.asarray(scaf).tolist(), np.asarray(start0).tolist(), np.asarray(length).tolist())):
        out[k] = mask(_ascii(seqs[c])[s:s + n], **p)[0]
    return out


def map_filter(tab_text: str, gff_text: str, agenome: Dict[str, object], maxtandem: float, params: Dict[str, int] = None,
               minLen=100, minIdt=90) -> Tuple[str, str]:
    """The tandem filter of `mimeo map` on the outputs of the oracle pipeline (lastz_oracle.mimeo_map): returns (GFF3 with the
    rows whose span [start1-1, end1) is masked more than maxtandem percent removed, TAB_HEADER + the .tab lines of the
    surviving rows in GFF order). Rows keep their UIDs; headers are unchanged."""
    # import_Align's row order with the raw lines kept: filter, then stable sort by (tName, tStart, tEnd, tStrand) as strings
    kept = []
    for line in tab_text.splitlines(True):
        f = line.strip().split()
        if line.strip().startswith('#') or not f:
            continue
        if int(f[3]) - int(f[2]) >= minLen and float(f[9]) >= minIdt:
            kept.append((f, line))
    kept.sort(key=lambda r: (r[0][0], r[0][2], r[0][3], r[0][1]))
    glines = gff_text.splitlines(True)
    head = [ln for ln in glines if ln.startswith('#')]
    rows = [ln for ln in glines if not ln.startswith('#')]
    assert len(rows) == len(kept), 'GFF rows and .tab rows disagree'
    p = dict(DEFAULTS, **(params or {}))
    out_rows, out_tab = [], []
    for row, (f, line) in zip(rows, kept):
        c = row.split('\t')
        assert (c[0], c[3], c[4]) == (f[0], f[2], f[3])
        s0, L = int(c[3]) - 1, int(c[4]) - int(c[3]) + 1
        m = mask(_ascii(agenome[c[0]])[s0:s0 + L], **p)[0]
        if not (100.0 * m / L > maxtandem):
            out_rows.append(row)
            out_tab.append(line if line.endswith('\n') else line + '\n')
    return ''.join(head + out_rows), ao.TAB_HEADER + ''.join(out_tab)
