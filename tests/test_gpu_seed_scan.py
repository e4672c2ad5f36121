"""GPU: the seed scan's survivor list (`mb2_test_seed_scan`), exactly. The HSP and alignment tests forgive the scan's mistakes
(an extra survivor is re-extended and dropped; a missing one is often covered by the next leader on its diagonal), so here
the sorted survivors and all four counters of seed_scan_kernel are held to tests/scan_reference.py, the exact statement of
its first stage, over the x-drop / threshold / transition grid, and the seed-hit and leader counters of the product paths
are held to the oracle's Stats."""
import numpy as np
import pytest

from tests import scan_reference as R
from tests.test_scan_reference import oracle_counts

pytestmark = pytest.mark.gpu

CASES = [('repeats', '+'), ('repeats', '-'), ('soft', '+'), ('edges', '+'), ('dense', '+'), ('family', '+')]
_DEV, _REF = {}, {}


@pytest.fixture(scope='module')
def G():
    from mimeo_b200 import genome
    return genome


def genomes(G, kind, strand):
    """(device T, device Q, reference T, reference Q), built once per module."""
    if (kind, strand) not in _DEV:
        g = R.scan_genome(kind)
        T = G.Genome.from_dict(g)
        TS = R.Space.from_ascii(list(g.values()))
        if strand == '+':
            _DEV[kind, strand] = (T, T, TS, TS)
        else:
            _DEV[kind, strand] = (T, T.revcomp(), TS, R.Space.from_ascii(list(g.values()), revcomp=True))
    return _DEV[kind, strand]


def sorted_rows(surv):
    return surv[np.lexsort((surv[:, 1], surv[:, 0]))] if len(surv) else surv.reshape(0, 2)


# At X = 6399 every run leader of these genomes is still open after its 60 / 90 columns, so every leader survives whatever K
# is: those rows check the always-open path and the cell count, not the threshold rule (X = 251 and 910 do).
@pytest.mark.parametrize('X', [251, 910, 6399])
@pytest.mark.parametrize('transition', [0, 1])
@pytest.mark.parametrize('kind,strand', CASES)
def test_survivors_and_counters_equal_reference(G, kind, strand, transition, X):
    T, Q, TS, QS = genomes(G, kind, strand)
    key = (kind, strand, transition)
    if key not in _REF:
        _REF[key] = R.leaders(TS, QS, transition)
    fs = R.first_stage(TS, QS, X, transition, lead=_REF[key])
    for K in (1000, 3000, 9000):
        surv, t_off, q_off, counters = G.test_seed_scan(T, Q, G.align_params(K, xdrop=X, transition=transition))
        assert t_off.tolist() == TS.off.tolist() and q_off.tolist() == QS.off.tolist()
        want, want_counters = R.summary(fs, K)
        assert counters == want_counters, (K, counters, want_counters)
        got = sorted_rows(surv)
        assert got.shape == want.shape and (got == want).all(), K
        assert len(want) > 0


def test_overflow_and_rescan_give_the_same_survivors(G):
    """An initial survivor capacity of 1: the scan overflows (every append past slot 0 is dropped by the capacity guard),
    scan_chunk grows the buffer and rescans; the result equals the default run."""
    T, Q, _, _ = genomes(G, 'family', '+')
    p = G.align_params(3000)
    a, _, _, ca = G.test_seed_scan(T, Q, p)
    b, _, _, cb = G.test_seed_scan(T, Q, p, init_cap=1)
    assert ca == cb and ca[0] > 1000
    assert (sorted_rows(a) == sorted_rows(b)).all()


@pytest.mark.parametrize('kind', R.SCAN_GENOMES)
def test_product_path_counters_equal_oracle_stats(G, kind):
    """seed_hits and leaders are defined exactly like the oracle's Stats.seed_hits / Stats.leaders: equal, summed over the
    scaffold pairs, through test_hsps (one strand) and through align (both strands)."""
    from mimeo_b200 import align as A
    T, _, _, _ = genomes(G, kind, '+')
    g = R.scan_genome(kind)
    for transition in (0, 1):
        p = G.align_params(3000, transition=transition)
        plus = oracle_counts(g, g, transition, '+')
        minus = oracle_counts(g, g, transition, '-')
        _, st = G.test_hsps(T, T, p)
        assert (int(st[1]), int(st[2])) == plus, transition
        _, st2 = A.align(T, T, p)
        assert (st2['seed_hits'], st2['leaders']) == (plus[0] + minus[0], plus[1] + minus[1]), transition
