"""The tandem-repeat report on the GPU (mb2_tandem_report) against the report oracle (tests/tandem_report_oracle.c) on every
field of every run, with its masked counts and runs against mb2_tandem_mask_runs from the same spans; and `mimeo filter
--reportTRF` / `mimeo map --maxtandem --reportTRF` end to end against the oracle pipelines."""
import numpy as np
import pytest

from oracle import lastz_oracle as lo
from oracle import tandem_oracle as to
from tests import tandem_report_reference as trr
from tests.test_tandem_emu import planted, random_seq

pytestmark = pytest.mark.gpu


def genome(seqs):
    from mimeo_b200 import genome as G
    return G.Genome([f's{k}' for k in range(len(seqs))], [np.frombuffer(s, np.uint8) for s in seqs])


def check(seqs, spans, mask_oracle=True, **p):
    """masked_reports against masked_runs and, per distinct run, the report oracle; with mask_oracle also the runs against the
    mask oracle. Returns the number of runs."""
    from mimeo_b200 import tandem
    prm = dict(to.DEFAULTS, **p)
    g = genome(seqs)
    try:
        scaf, st, ln = (np.array([s[k] for s in spans], np.int64) for k in range(3))
        m, reps = tandem.masked_reports(g, scaf, st, ln, prm)
        m_runs, runs = tandem.masked_runs(g, scaf, st, ln, prm)
    finally:
        g.close()
    assert (m == m_runs).all()
    cache, want_mask = {}, {}
    for k, (c, s, n) in enumerate(spans):
        assert [(r.start, r.end) for r in reps[k]] == runs[k], f'span {k}: report runs differ from mb2_tandem_mask_runs'
        if mask_oracle:
            if (c, s, n) not in want_mask:
                want_mask[(c, s, n)] = to.mask(seqs[c][s:s + n], **prm)
            assert (int(m[k]), runs[k]) == want_mask[(c, s, n)]
        for r in reps[k]:
            key = (c, s + r.start, r.end - r.start + 1)
            if key not in cache:
                cache[key] = trr.report(seqs[c][key[1]:key[1] + key[2]], **prm)
            assert tuple(r[2:]) == cache[key], f'span {k} run {r[:2]} {prm}: gpu {tuple(r[2:])} != oracle {cache[key]}'
    return sum(len(v) for v in reps)


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
    assert check(seqs, spans) > 50


@pytest.mark.parametrize('P', [1, 7, 50, 64, 100, 256])
def test_periods_and_shift_counts(P):
    rng = np.random.default_rng(P)
    seqs = [planted(rng, 4 * P + 300, int(rng.integers(1, P + 1)), 6, sub=0.03) for _ in range(12)]
    for _ in range(4):                                                  # soft-masked arrays with N, long enough to be masked at any P
        d = int(rng.integers(1, min(P, 31) + 1))
        seqs.append(planted(rng, 600, d, max(30.0, 150 / d), sub=0.02, lower=True, ns=2))
    spans = [(k, 0, len(s)) for k, s in enumerate(seqs)]
    assert check(seqs, spans, maxperiod=P) > 0


def test_non_default_scores_and_16_bit_storage():
    rng = np.random.default_rng(5)
    seqs = [planted(rng, 900, int(rng.integers(1, 30)), 20, sub=0.05) for _ in range(10)]
    spans = [(k, 0, len(s)) for k, s in enumerate(seqs)]
    assert check(seqs, spans, match=3, mismatch=4, delta=2, minscore=30, maxperiod=33) > 0
    assert check(seqs, spans, match=5, mismatch=11, delta=9, minscore=400, maxperiod=20) > 0     # minscore + mismatch > 255


def test_run_over_100_kbp():
    rng = np.random.default_rng(6)
    arr = planted(rng, 0, 37, 130_000 / 37, sub=0.01)
    big = random_seq(rng, 3000) + arr + random_seq(rng, 2000)
    n = check([big], [(0, 0, len(big)), (0, 1000, 120_000)], mask_oracle=False, maxperiod=100)
    from mimeo_b200 import tandem
    g = genome([big])
    try:
        _m, reps = tandem.masked_reports(g, [0], [0], [len(big)], dict(to.DEFAULTS, maxperiod=100))
    finally:
        g.close()
    longest = max(reps[0], key=lambda r: r.end - r.start)
    assert n >= 1 and longest.end - longest.start + 1 > 100_000 and longest.period == 37


def test_thousands_of_runs_in_one_call():
    rng = np.random.default_rng(8)
    chunks = []
    for k in range(3000):
        d = int(rng.integers(1, 60))
        chunks.append(planted(rng, 260, d, max(3.0, 80 / d), sub=float(rng.choice([0, 0.03])), lower=k % 7 == 0, ns=int(k % 5 == 0)))
    seq = b''.join(chunks)
    offs = np.cumsum([0] + [len(c) for c in chunks])
    spans = [(0, int(offs[k]), int(offs[k + 1] - offs[k])) for k in range(len(chunks))] + [(0, 0, int(offs[-1]) // 2)]
    assert check([seq], spans, mask_oracle=False, maxperiod=64) > 2500


def test_refusals_match_the_mask():
    from mimeo_b200 import _lib, tandem
    seqs = [np.frombuffer(b'ACGT' * 100, np.uint8)]
    for bad in (dict(maxperiod=257), dict(maxperiod=0), dict(match=0), dict(minscore=65530, mismatch=7), dict(delta=-1)):
        with pytest.raises(_lib.Mb2Error) as e:
            tandem.masked_reports(seqs, [0], [0], [400], dict(to.DEFAULTS, **bad))
        assert e.value.code == -2
    with pytest.raises(_lib.Mb2Error):
        tandem.masked_reports(seqs, [0], [350], [51], to.DEFAULTS)


def test_filter_cli_report_on_gpu(tmp_path, monkeypatch):
    from tests.test_filter_cli import fasta_text, library, run_cli
    text = fasta_text(library())
    (tmp_path / 'lib.fa').write_bytes(text)
    base = ['filter', '--infile', str(tmp_path / 'lib.fa'), '--outfile', 'lib.fa', '--writeTRF']
    assert run_cli(monkeypatch, base + ['-d', str(tmp_path / 'a')]) == 0
    assert run_cli(monkeypatch, base + ['-d', str(tmp_path / 'b'), '--reportTRF']) == 0
    got = (tmp_path / 'b' / 'lib_TRF.gff3').read_text()
    assert got == trr.fasta_text_report(text.decode()) and got.count('\n') > 10
    for name in ('lib.fa', 'lib_TRFmasked.fa'):
        assert (tmp_path / 'a' / name).read_bytes() == (tmp_path / 'b' / name).read_bytes()


def test_map_cli_report_on_gpu(tmp_path, monkeypatch):
    from tests.test_host_api import _write_genome
    from tests.test_tandem_cli import map_inputs, run_cli
    a, b = map_inputs()
    monkeypatch.chdir(tmp_path)
    _write_genome(tmp_path / 'a.fa', a)
    _write_genome(tmp_path / 'b.fa', b)
    base = ['map', '--afasta', 'a.fa', '--bfasta', 'b.fa', '--minIdt', '90', '--outfile', 'm.tab', '--gffout', 'm.gff3', '--maxtandem', '40',
            '--writeTRF']
    run_cli(monkeypatch, base)
    plain = {n: (tmp_path / n).read_bytes() for n in ('m.tab', 'm.gff3', 'm_TRFfiltered.tab')}
    run_cli(monkeypatch, base + ['--reportTRF'])
    _tab, gff = lo.mimeo_map({k: lo.encode(v) for k, v in a.items()}, {k: lo.encode(v) for k, v in b.items()}, minIdt=90, minLen=100)
    assert (tmp_path / 'm_TRF.gff3').read_text() == trr.map_report(gff, {k: v.tobytes() for k, v in a.items()})
    assert {n: (tmp_path / n).read_bytes() for n in plain} == plain
