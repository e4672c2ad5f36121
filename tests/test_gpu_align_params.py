"""GPU parity of the whole alignment stage away from mimeo's defaults: the edges of the x-drop, threshold, y-drop and gap
ranges the C ABI accepts, every row against the oracle; the pad between two scaffolds at the largest accepted x-drop; and
values outside the ranges, which must fail with an error instead of running."""
import numpy as np
import pytest

from oracle import lastz_oracle as lo
from tests.helpers import synth_genome
from tests.test_gpu_align import gpu_rows, oracle_rows

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def M():
    import mimeo_b200.align as A
    import mimeo_b200.genome as G
    return A, G


@pytest.fixture(scope='module')
def small():
    return synth_genome(81, 2, 15_000, 3, copies=(3, 5), fam_len=(300, 1500), sub=0.10, indel=0.008, n_runs=2)


@pytest.mark.parametrize('xdrop', [251, 6399])
def test_xdrop_edges(M, xdrop):
    A, G = M
    g = synth_genome(82, 3, 25_000, 3, copies=(3, 6), fam_len=(300, 2000), sub=0.10, indel=0.006, n_runs=3)
    T = G.Genome.from_dict(g)
    hits, _ = A.align(T, T, G.align_params(3000, xdrop=xdrop))
    want = oracle_rows(g, g, lo.default_params(3000, xdrop=xdrop))
    assert gpu_rows(hits) == want and len(want) > 10


@pytest.mark.parametrize('hspthresh,gappedthresh', [(1500, 2500), (1500, 1000), (6000, 8000), (6000, 4500)])
def test_hspthresh_and_gappedthresh_apart(M, hspthresh, gappedthresh):
    A, G = M
    g = synth_genome(83, 3, 25_000, 3, copies=(3, 6), fam_len=(300, 2000), sub=0.10, indel=0.006, n_runs=2)
    T = G.Genome.from_dict(g)
    hits, _ = A.align(T, T, G.align_params(hspthresh, gappedthresh=gappedthresh))
    want = oracle_rows(g, g, lo.default_params(hspthresh, gappedthresh=gappedthresh))
    assert gpu_rows(hits) == want and len(want) > 5


@pytest.mark.parametrize('ydrop', [1000, 20000])
@pytest.mark.parametrize('gap_open', [0, 2000])
@pytest.mark.parametrize('gap_extend', [10, 60])
def test_ydrop_and_gap_corners(M, small, ydrop, gap_open, gap_extend):
    """At y-drop 20000 with cheap gaps some extensions of this genome keep more than 2048 diagonals alive, more than the wide
    kernel holds: they take the full-row fallback of the gapped stage."""
    A, G = M
    T = G.Genome.from_dict(small)
    kw = dict(ydrop=ydrop, gap_open=gap_open, gap_extend=gap_extend)
    hits, _ = A.align(T, T, G.align_params(3000, **kw))
    want = oracle_rows(small, small, lo.default_params(3000, **kw))
    assert gpu_rows(hits) == want and len(want) > 5


def pad_genomes(G):
    """Two separate genome objects with identical scaffolds of 6400 and 6451 bases: the first is followed by a pad of exactly
    64 columns, so the main diagonal of the two copies runs scaffold, 64 pad columns, scaffold."""
    rng = np.random.default_rng(84)
    acgt = np.frombuffer(b'ACGT', dtype=np.uint8)
    g = {'s0': acgt[rng.integers(0, 4, 6400)].copy(), 's1': acgt[rng.integers(0, 4, 6451)].copy()}
    return g, G.Genome.from_dict(g), G.Genome.from_dict({k: v.copy() for k, v in g.items()})


def test_pad_between_scaffolds_at_the_largest_xdrop(M):
    A, G = M
    g, T, Q = pad_genomes(G)
    hits, _ = A.align(T, Q, G.align_params(3000, xdrop=6399))
    want = oracle_rows(g, g, lo.default_params(3000, xdrop=6399))
    assert gpu_rows(hits) == want
    assert {(r[0], r[1], r[2], r[3], r[4]) for r in want} >= {(0, 0, 0, 1, 6400), (1, 1, 0, 1, 6451)}
    hsps, _ = G.test_hsps(T, Q, G.align_params(3000, xdrop=6399))
    assert max(hsps[:, 3]) == 6451


@pytest.mark.parametrize('kw', [dict(xdrop=6400), dict(xdrop=7000), dict(xdrop=250), dict(xdrop=0), dict(ydrop=999),
                                dict(ydrop=20001), dict(gap_open=-1), dict(gap_open=2001), dict(gap_extend=9),
                                dict(gap_extend=61), dict(hspthresh=0)])
def test_parameters_outside_the_range_are_rejected(M, kw):
    """Rejected up front by every entry point, even when no stage would have reached the check that depends on the value."""
    A, G = M
    from mimeo_b200 import _lib
    _, T, Q = pad_genomes(G)
    p = G.align_params(3000)
    for k, v in kw.items():
        setattr(p, k, v)
    with pytest.raises(_lib.Mb2Error) as e:
        A.align(T, Q, p)
    assert e.value.code == -2
    with pytest.raises(_lib.Mb2Error):
        G.test_hsps(T, Q, p)
    with pytest.raises(_lib.Mb2Error):
        G.test_seed_scan(T, Q, p)
    tiny = G.Genome.from_dict({'a': np.frombuffer(b'ACGT' * 4, dtype=np.uint8)})     # no seed at all: nothing would run
    with pytest.raises(_lib.Mb2Error):
        A.align(tiny, tiny, p)
