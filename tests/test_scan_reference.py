"""CPU checks of tests/scan_reference.py, the exact statement of the seed scan's first stage that the GPU survivor test
(tests/test_gpu_seed_scan.py) holds the kernel to. No GPU needed:
  * its seed-hit and run-leader counts, summed over the scaffold pairs, equal the LASTZ-restatement oracle's Stats;
  * its vectorised extension agrees with a plain per-hit loop, hit for hit, including hits at scaffold edges."""
import numpy as np
import pytest

from oracle import lastz_oracle as lo
from tests import scan_reference as R


def oracle_counts(tg, qg, transition, strand='+'):
    """Seed hits and leaders of the oracle summed over every (target scaffold, query scaffold) pair of one strand."""
    st = lo.Stats()
    p = lo.default_params(3000, transition=transition)
    for t in tg.values():
        tix = lo.TargetIndex(lo.encode(t))
        for q in qg.values():
            qc = lo.encode(q)
            lo.hsps(tix, qc if strand == '+' else lo.revcomp_codes(qc), p, st)
    return st.seed_hits, st.leaders


@pytest.mark.parametrize('kind', R.SCAN_GENOMES)
@pytest.mark.parametrize('transition', [0, 1])
def test_reference_counts_equal_oracle_stats(kind, transition):
    g = R.scan_genome(kind)
    T = R.Space.from_ascii(list(g.values()))
    for strand in ('+', '-') if kind in ('repeats', 'soft') else ('+',):
        Q = T if strand == '+' else R.Space.from_ascii(list(g.values()), revcomp=True)
        nhits, I, J = R.leaders(T, Q, transition)
        want = oracle_counts(g, g, transition, strand)
        assert (nhits, len(I)) == want, (strand, (nhits, len(I)), want)
        assert want[1] > 100


def test_reference_x_mode_and_soft_mask_on_one_side():
    """Two different genomes, one of them soft-masked: hits need both windows seedable."""
    a = R.scan_genome('repeats')
    b = R.scan_genome('soft')
    b['scaf000'][3000:5000] = a['scaf001'][1000:3000] | 0x20
    b['scaf001'][7000:9000] = a['scaf002'][4000:6000]
    for transition in (0, 1):
        nhits, I, J = R.leaders(R.Space.from_ascii(list(a.values())), R.Space.from_ascii(list(b.values())), transition)
        assert (nhits, len(I)) == oracle_counts(a, b, transition)


def test_layout_matches_the_device_rule():
    off, G = R.layout([6400, 6451, 6463, 1, 64, 65])
    assert off.tolist() == [2048, 8512, 15040, 21568, 21696, 21824] and G == 22016 + 2048
    gaps = np.diff(off) - np.array([6400, 6451, 6463, 1, 64])
    assert gaps.min() == 64 and gaps.tolist()[:3] == [64, 77, 65]


@pytest.mark.parametrize('kind', ['edges', 'repeats', 'family'])
@pytest.mark.parametrize('X', [251, 910, 6399])
def test_vectorised_extension_equals_per_hit_loop(kind, X):
    g = R.scan_genome(kind)
    T = R.Space.from_ascii(list(g.values()))
    Q = R.Space.from_ascii(list(g.values()), revcomp=kind == 'repeats')
    transition = 1
    I, J = R.seed_hits(T, Q, transition)
    lead = R.is_leader(T, Q, I, J, transition)
    rng = np.random.default_rng(X)
    # a few hundred hits: random hits, random leaders, and leaders whose extension reaches a scaffold edge within its 60 / 90
    # columns
    ts, qs = T.scaffold_of(I), Q.scaffold_of(J)
    near = (T.scaffold_of(I + 79) != ts) | (T.scaffold_of(I - 72) != ts) | (Q.scaffold_of(J + 79) != qs) | (Q.scaffold_of(J - 72) != qs)
    li = np.flatnonzero(lead)
    pick = np.unique(np.concatenate([rng.choice(len(I), min(100, len(I)), replace=False), rng.choice(li, min(200, len(li)), replace=False),
                                     np.flatnonzero(near & lead)[:150]]))
    assert kind != 'edges' or (near & lead)[pick].sum() >= 50
    fs = R.first_stage(T, Q, X, transition, lead=(len(I), I[pick][lead[pick]], J[pick][lead[pick]]))
    row = {(i, j): k for k, (i, j) in enumerate(zip(fs['i'].tolist(), fs['j'].tolist()))}
    checked = 0
    for i, j in zip(I[pick].tolist(), J[pick].tolist()):
        is_lead, br, open_r, bl, open_l, chunks = R.brute_hit(T, Q, i, j, X, transition)
        assert is_lead == ((i, j) in row)
        if not is_lead:
            continue
        k = row[(i, j)]
        got = (int(fs['best_r'][k]), bool(fs['tcol_r'][k] >= R.RIGHT_COLS), int(fs['best_l'][k]), bool(fs['tcol_l'][k] >= R.LEFT_COLS),
               int(fs['chunks'][k]))
        assert got == (br, open_r, bl, open_l, chunks), (i, j)
        checked += 1
    assert checked >= 50


def test_gpu_genomes_reach_the_scan_paths():
    """The genomes of tests/test_gpu_seed_scan.py reach what they are there for. A warp takes whole rounds of 32 query
    positions, so the hits one round defers all go to one warp's queue of 64 records: a round that defers more than 64
    wraps the queue around and drains it more than once, and one whose count is not a multiple of 32 leaves a partial drain.
    The dense genome puts thousands of hits on one query position (full descriptor steps of 96); the edge genome has hits at
    both ends of scaffolds and a query whose last round of 32 positions is partial."""
    fam = R.scan_genome('family')
    S = R.Space.from_ascii(list(fam.values()))
    fs = R.first_stage(S, S, 910, 1)
    d = R.deferred(fs)
    per_round = np.bincount((fs['j'][d] - S.off[0]) // 32)
    assert d.sum() > 10_000 and (per_round > 64).sum() > 20 and (per_round % 32 != 0).sum() > 20
    # hits still open after right window 0 but closed after left window 1, and the other way round
    assert ((fs['tcol_r'] >= 30) & (fs['tcol_l'] < 60)).sum() > 100 and ((fs['tcol_r'] < 30) & (fs['tcol_l'] >= 60)).sum() > 100

    dense = R.scan_genome('dense')
    S = R.Space.from_ascii(list(dense.values()))
    _, J = R.seed_hits(S, S, 0)
    assert np.bincount(J).max() > 900

    edges = R.scan_genome('edges')
    S = R.Space.from_ascii(list(edges.values()))
    assert (S.off[-1] + S.len[-1] - S.off[0]) % 32 != 0
    assert [n % 64 for n in S.len[:3].tolist()] == [0, 51, 63]
    _, I, J = R.leaders(S, S, 1)
    for n in (18, 19, 20, 63, 64, 65):
        s = list(edges).index(f'head{n}')
        assert (S.scaffold_of(J) == s).any() == (n >= 19), n
