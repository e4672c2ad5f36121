"""The tandem-repeat mask on the GPU (mb2_tandem_mask / mb2_test_tandem_mask) against the C oracle, span by span: masked
count and every merged masked run; and `mimeo map --maxtandem --writeTRF` end to end against the oracle pipeline."""
import numpy as np
import pytest

from oracle import lastz_oracle as lo
from oracle import tandem_oracle as to
from tests.test_tandem_emu import planted, random_seq

pytestmark = pytest.mark.gpu


def genome(seqs):
    from mimeo_b200 import genome as G
    return G.Genome([f's{k}' for k in range(len(seqs))], [np.frombuffer(s, np.uint8) for s in seqs])


def check(seqs, spans, budget=0, **p):
    from mimeo_b200 import tandem
    prm = dict(to.DEFAULTS, **p)
    g = genome(seqs)
    try:
        scaf, st, ln = (np.array([s[k] for s in spans], np.int64) for k in range(3))
        got_m, got_iv = tandem.masked_runs(g, scaf, st, ln, prm, budget)
        cnt = tandem.masked_counts(g, scaf, st, ln, prm)
    finally:
        g.close()
    assert (cnt == got_m).all()
    cache = {}
    for k, (c, s, n) in enumerate(spans):
        if (c, s, n) not in cache:
            cache[(c, s, n)] = to.mask(seqs[c][s:s + n], **prm)
        want = cache[(c, s, n)]
        assert (int(got_m[k]), got_iv[k]) == want, f'span {k} ({c}, {s}, {n}) {prm}: gpu {int(got_m[k])} {got_iv[k][:5]} != oracle {want[0]} {want[1][:5]}'
    return int(got_m.sum())


def test_planted_periods_edges_n_runs_soft_mask_and_duplicates():
    rng = np.random.default_rng(9)
    seqs, spans = [], []
    for period in range(1, 51):
        s = planted(rng, 600, period, max(3.0, 120 / period), sub=float(rng.choice([0, 0.02, 0.05])), lower=period % 3 == 0,
                    ns=period % 4)
        seqs.append(s)
        spans += [(period - 1, 0, len(s)), (period - 1, 0, 150), (period - 1, len(s) - 200, 200), (period - 1, 100, 380)]
    seqs.append(b'N' * 40 + b'AC' * 60 + b'N' * 70 + b'ACGTT' * 30 + b'NNNN')
    spans += [(50, 0, len(seqs[-1])), (50, 30, 200), (50, 5, 0), (50, 7, 1), (50, 9, 2)]
    spans += spans[:40]                                                 # duplicated spans
    assert check(seqs, spans) > 0


@pytest.mark.parametrize('P', [1, 7, 50, 64, 100, 256])
def test_periods_and_layouts(P):
    rng = np.random.default_rng(P)
    seqs = [planted(rng, 4 * P + 300, int(rng.integers(1, P + 1)), 6, sub=0.03) for _ in range(12)]
    spans = [(k, 0, len(s)) for k, s in enumerate(seqs)]
    check(seqs, spans, maxperiod=P)


def test_non_default_scores_and_16_bit_storage():
    rng = np.random.default_rng(5)
    seqs = [planted(rng, 900, int(rng.integers(1, 30)), 20, sub=0.05) for _ in range(10)]
    spans = [(k, 0, len(s)) for k, s in enumerate(seqs)]
    check(seqs, spans, match=3, mismatch=4, delta=2, minscore=30, maxperiod=33)
    check(seqs, spans, match=5, mismatch=11, delta=9, minscore=400, maxperiod=20)     # minscore + mismatch > 255


def test_long_spans_and_many_launches():
    rng = np.random.default_rng(6)
    big = bytearray(random_seq(rng, 520_000))
    for at in range(1000, 510_000, 37_000):
        arr = planted(rng, 0, int(rng.integers(1, 50)), float(rng.uniform(5, 40)), sub=0.03)
        big[at:at + len(arr)] = arr
    big = bytes(big)
    seqs = [big]
    spans = [(0, 0, len(big)), (0, 3, 70_001), (0, 200_000, 66_000)]
    spans += [(0, int(x), int(rng.integers(100, 3000))) for x in rng.integers(0, 500_000, 60)]
    check(seqs, spans)
    check(seqs, spans[1:], budget=8 << 20)       # a small storage bound: many launches, the 70 kbp span alone in one


def test_parameters_beyond_the_cap_are_refused():
    from mimeo_b200 import _lib, tandem
    g = genome([b'ACGT' * 100])
    try:
        one = (np.zeros(1, np.int32), np.zeros(1, np.int64), np.full(1, 100, np.int64))
        for bad in (dict(maxperiod=257), dict(maxperiod=0), dict(match=0), dict(minscore=65530, mismatch=7), dict(delta=-1)):
            with pytest.raises(_lib.Mb2Error) as e:
                tandem.masked_counts(g, *one, dict(to.DEFAULTS, **bad))
            assert e.value.code == -2
        with pytest.raises(_lib.Mb2Error):
            tandem.masked_counts(g, np.zeros(1, np.int32), np.full(1, 350, np.int64), np.full(1, 51, np.int64), to.DEFAULTS)
    finally:
        g.close()


def test_map_maxtandem_writetrf_on_gpu_matches_oracle_pipeline(tmp_path, monkeypatch):
    from tests.test_host_api import _write_genome
    from tests.test_tandem_cli import map_inputs, run_cli
    a, b = map_inputs()
    monkeypatch.chdir(tmp_path)
    _write_genome(tmp_path / 'a.fa', a)
    _write_genome(tmp_path / 'b.fa', b)
    run_cli(monkeypatch, ['map', '--afasta', 'a.fa', '--bfasta', 'b.fa', '--minIdt', '90', '--outfile', 'm.tab', '--gffout', 'm.gff3',
                          '--maxtandem', '40', '--writeTRF'])
    tab, gff = lo.mimeo_map({k: lo.encode(v) for k, v in a.items()}, {k: lo.encode(v) for k, v in b.items()}, minIdt=90, minLen=100)
    want_gff, want_tab = to.map_filter(tab, gff, {k: v.tobytes() for k, v in a.items()}, 40.0, minLen=100, minIdt=90)
    assert (tmp_path / 'm.tab').read_text() == tab
    assert (tmp_path / 'm.gff3').read_text() == want_gff and want_gff != gff
    assert (tmp_path / 'm_TRFfiltered.tab').read_text() == want_tab
