"""Device-resident genomes (host mirror of what `splitFasta` + LASTZ's reader do for the reference:
utils.py:274-309). Sequences are plain ASCII; packing to 2 bits + N-mask happens on the GPU."""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Sequence

import numpy as np

from . import _lib


def _as_ascii(seq) -> np.ndarray:
    if isinstance(seq, str):
        seq = seq.encode()
    if isinstance(seq, (bytes, bytearray)):
        return np.frombuffer(bytes(seq), dtype=np.uint8)
    a = np.ascontiguousarray(seq, dtype=np.uint8)
    return a


class Genome:
    """names[i] / lengths[i] describe scaffold i; `handle` is the opaque mb2_genome*."""

    def __init__(self, names: Sequence[str], seqs: Sequence, _handle=None, _lengths=None):
        _lib.init()
        self.names: List[str] = list(names)
        if _handle is not None:
            self.handle = _handle
            self.lengths = list(_lengths)
            return
        arrs = [_as_ascii(s) for s in seqs]
        if len(arrs) != len(self.names) or not arrs:
            raise ValueError('need one sequence per name and at least one scaffold')
        self.lengths = [int(len(a)) for a in arrs]
        ptrs = (C.c_void_p * len(arrs))(*[a.ctypes.data for a in arrs])
        lens = np.array(self.lengths, dtype=np.uint64)
        h = C.c_void_p()
        _lib.check(_lib.lib().mb2_genome_create(ptrs, lens.ctypes.data, len(arrs), C.byref(h)))
        self.handle = h

    @classmethod
    def from_dict(cls, d: Dict[str, object]) -> 'Genome':
        names = list(d)
        return cls(names, [d[n] for n in names])

    def revcomp(self) -> 'Genome':
        h = C.c_void_p()
        _lib.check(_lib.lib().mb2_genome_revcomp(self.handle, C.byref(h)))
        return Genome(self.names, None, _handle=h, _lengths=self.lengths)

    def both_strands(self) -> 'Genome':
        """Scaffolds followed by their reverse complements (2n scaffolds): the companion mb2_align takes for strands=3."""
        h = C.c_void_p()
        _lib.check(_lib.lib().mb2_genome_both_strands(self.handle, C.byref(h)))
        return Genome(self.names + [n + '(-)' for n in self.names], None, _handle=h, _lengths=self.lengths + self.lengths)

    def decode(self, scaf: int) -> np.ndarray:
        out = np.zeros(self.lengths[scaf], dtype=np.uint8)
        _lib.check(_lib.lib().mb2_genome_decode(self.handle, scaf, out.ctypes.data))
        return out

    def nibbles(self) -> np.ndarray:
        """Test hook: the 4-bit code of every padded position (uint8 per position, the device plane unpacked)."""
        n = C.c_uint64(0)
        _lib.check(_lib.lib().mb2_test_genome_nibbles(self.handle, None, 0, C.byref(n)))
        words = np.zeros(int(n.value), dtype=np.uint32)
        _lib.check(_lib.lib().mb2_test_genome_nibbles(self.handle, words.ctypes.data, len(words), C.byref(n)))
        return ((words[:, None] >> (4 * np.arange(8, dtype=np.uint32))) & 15).astype(np.uint8).reshape(-1)

    def close(self):
        if getattr(self, 'handle', None):
            _lib.lib().mb2_genome_free(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def align_params(hspthresh=3000, **kw) -> _lib.AlignParams:
    p = _lib.AlignParams()
    _lib.lib().mb2_default_align_params(C.byref(p))
    p.hspthresh = int(hspthresh)
    p.gappedthresh = int(hspthresh)
    for k, v in kw.items():
        setattr(p, k, int(v))
    return p


def test_hsps(T: Genome, Q: Genome, p: _lib.AlignParams):
    """Stage (a)+(b) only (test hook). Returns (array (n,5) [tile,s1,s2,len,score], stats[16])."""
    h = _lib.Hsps()
    stats = np.zeros(16, dtype=np.uint64)
    _lib.check(_lib.lib().mb2_test_hsps(T.handle, Q.handle, C.byref(p), C.byref(h), stats.ctypes.data))
    try:
        n = int(h.n)
        cols = [np.ctypeslib.as_array(x, shape=(n,)).astype(np.int64) if n else np.zeros(0, np.int64)
                for x in (h.tile, h.s1, h.s2, h.len, h.score)]
        out = np.stack(cols, axis=1) if n else np.zeros((0, 5), np.int64)
    finally:
        _lib.lib().mb2_free_hsps(C.byref(h))
    return out, stats


def test_seed_scan(T: Genome, Q: Genome, p: _lib.AlignParams, init_cap: int = 0):
    """Stage (a) only (test hook): the seed hits the first-stage x-drop could not rule out, in one scan of the whole query.
    Returns (survivors (n,2) [target, query] padded seed starts in scan order, t_off, q_off, counters[4] = survivors,
    seed hits, leaders, stage-1 cells). init_cap: initial survivor capacity (0 = default)."""
    s = _lib.SeedSurvivors()
    _lib.check(_lib.lib().mb2_test_seed_scan(T.handle, Q.handle, C.byref(p), int(init_cap), C.byref(s)))
    try:
        n = int(s.n)
        surv = np.zeros((n, 2), np.int64)
        if n:
            surv[:, 0] = np.ctypeslib.as_array(s.t_pos, shape=(n,))
            surv[:, 1] = np.ctypeslib.as_array(s.q_pos, shape=(n,))
        t_off = np.ctypeslib.as_array(s.t_off, shape=(int(s.t_nscaf),)).astype(np.int64)
        q_off = np.ctypeslib.as_array(s.q_off, shape=(int(s.q_nscaf),)).astype(np.int64)
        counters = [int(x) for x in s.counters]
    finally:
        _lib.lib().mb2_free_seed_survivors(C.byref(s))
    return surv, t_off, q_off, counters
