"""Bands wider than the widest layout of the y-drop kernel, on the CPU warp emulator. At y-drop 20000 with cheap gaps, an
extension from an anchor inside a repeat pair keeps more than 2048 diagonals alive on one anti-diagonal; the wide kernel
then returns ST_BAND and the gapped stage reruns the item with the full-row fallback (ydrop_full_warp, same source file).
Held to the oracle's ydrop_extend: the anchor where this was first seen, and every alignment anchor of a small repeat genome
at the three penalty corners where it happens, each taken through the same narrow -> wide -> full-row sequence as
gapped.cu."""
import ctypes as C

import numpy as np
import pytest

from oracle import lastz_oracle as lo
from tests.helpers import synth_genome
from tests.test_ydrop_emu import emu_ext, emu_lib, kernel_codes, oracle_ext, PAD

ST_OK, ST_WIDE, ST_BAND = 0, 2, 4
CORNERS = [(20000, 0, 60), (20000, 0, 10), (20000, 2000, 10)]


def full_lib():
    l = emu_lib()
    l.emu_full.restype = C.c_int
    l.emu_full.argtypes = [C.c_void_p, C.c_void_p, C.c_long, C.c_long, C.c_int, C.c_long, C.c_long, C.c_int, C.c_int, C.c_int, C.c_long,
                           C.c_void_p]
    return l


def gapped_stage_ext(l, t, tk, a1, q, qk, a2, d, p):
    """One extension as the gapped stage runs it: common kernel, wide rerun, full-row rerun. Returns (result[:5], path)."""
    got = emu_ext(l, tk, a1, qk, a2, d, p, 32)
    path = 'narrow'
    if got[5] == ST_WIDE:
        got, path = emu_ext(l, tk, a1, qk, a2, d, p, 64), 'wide'
    if got[5] == ST_BAND:
        tn, qn = (len(t) - a1, len(q) - a2) if d > 0 else (a1, a2)
        got = np.zeros(7, np.int32).tolist()
        out = np.zeros(7, np.int32)
        l.emu_full(tk.ctypes.data, qk.ctypes.data, PAD + a1, PAD + a2, d, tn, qn, p.gap_open, p.gap_extend, p.ydrop, 1 << 16, out.ctypes.data)
        got, path = out.tolist(), 'full'
    assert got[5] == ST_OK, (path, got)
    return got[:5], path


def small_genome():
    return synth_genome(81, 2, 15_000, 3, copies=(3, 5), fam_len=(300, 1500), sub=0.10, indel=0.008, n_runs=2)


def test_band_wider_than_the_wide_kernel_takes_the_full_rows():
    l = full_lib()
    g = small_genome()
    t, q = lo.encode(g['scaf000']), lo.encode(g['scaf001'])
    tk, qk = kernel_codes(t), kernel_codes(q)
    p = lo.default_params(3000, ydrop=20000, gap_open=0, gap_extend=60)
    paths = []
    for d in (+1, -1):
        want, _ = oracle_ext(t, 7513, q, 6128, d, p)
        got, path = gapped_stage_ext(l, t, tk, 7513, q, qk, 6128, d, p)
        assert got == want, (d, path)
        paths.append(path)
    assert 'full' in paths


@pytest.mark.parametrize('ydrop,gap_open,gap_extend', CORNERS)
def test_alignment_anchors_at_the_wide_band_corners(ydrop, gap_open, gap_extend):
    l = full_lib()
    g = small_genome()
    p = lo.default_params(3000, ydrop=ydrop, gap_open=gap_open, gap_extend=gap_extend)
    codes = {k: lo.encode(v) for k, v in g.items()}
    paths = []
    for tname, t in codes.items():
        tix = lo.TargetIndex(t)
        tk = kernel_codes(t)
        for qname, qc in codes.items():
            for strand in (0, 1):
                q = qc if strand == 0 else lo.revcomp_codes(qc)
                qk = kernel_codes(q)
                for a1, a2 in {(int(r[7]), int(r[8])) for r in lo.align_tile(tix, q, p).tolist()}:
                    for d in (+1, -1):
                        want, _ = oracle_ext(t, a1, q, a2, d, p)
                        got, path = gapped_stage_ext(l, t, tk, a1, q, qk, a2, d, p)
                        assert got == want, (tname, qname, strand, a1, a2, d, path)
                        paths.append(path)
    assert paths.count('full') >= 2, paths
