"""GPU: the 4-bit code plane (nb) that pack_kernel, revcomp_kernel and both_strands_kernel write next to the 2-bit pack,
against a numpy encoding of the same ASCII: base | parity << 2 for A, C, G, T in either case, 8 for N, IUPAC codes and every
pad position of the padded coordinate space."""
import numpy as np
import pytest

from tests import scan_reference as R

pytestmark = pytest.mark.gpu


def want_plane(S):
    return np.where(S.bad, 8, S.base | (((S.base ^ (S.base >> 1)) & 1) << 2)).astype(np.uint8)


def test_nibble_plane_equals_numpy_encoding():
    from mimeo_b200 import genome as G
    rng = np.random.default_rng(3)
    g = {}
    for k, n in enumerate((1, 63, 64, 65, 700, 2051)):
        s = np.frombuffer(b'ACGTacgtNRYKMSWnry', dtype=np.uint8)[rng.integers(0, 18, n)].copy()
        if n > 100:
            s[: n // 2] = np.frombuffer(b'ACGT', dtype=np.uint8)[rng.integers(0, 4, n // 2)]
        g[f's{k}'] = s
    seqs = list(g.values())
    T = G.Genome.from_dict(g)
    cases = [(T, R.Space.from_ascii(seqs)),
             (T.revcomp(), R.Space.from_ascii(seqs, revcomp=True)),
             (T.both_strands(), R.Space([R.lo.encode(s) for s in seqs] + [R.lo.revcomp_codes(R.lo.encode(s)) for s in seqs]))]
    for dev, S in cases:
        got = dev.nibbles()
        want = want_plane(S)
        assert got.shape == want.shape
        assert (got == want).all(), np.flatnonzero(got != want)[:10]
