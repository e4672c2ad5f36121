"""`mimeo filter` on the GPU: whole-record masks and runs from mb2_tandem_mask_runs against the C oracle, record by record,
and against mb2_tandem_mask / mb2_test_tandem_mask on the same input; refusals; and the CLI end to end against
filter_reference.fasta_filter."""
import numpy as np
import pytest

from oracle import tandem_oracle as to
from tests.test_filter_cli import check_outputs, fasta_text, library, run_cli
from tests.test_tandem_emu import planted, random_seq

pytestmark = pytest.mark.gpu


def n_run(rng, seq, k):
    """seq with a run of k N bases (upper or lower case) written into its middle third."""
    s = bytearray(seq)
    at = int(rng.integers(len(s) // 3, max(len(s) // 3 + 1, 2 * len(s) // 3 - k)))
    s[at:at + k] = (b'N' if rng.random() < 0.5 else b'n') * k
    return bytes(s[:len(seq)])


def check_records(seqs, **p):
    """record_masks with runs (mb2_tandem_mask_runs) against the oracle on every record; its counts against mb2_tandem_mask
    and its runs against mb2_test_tandem_mask on a Genome of the same records. Returns the total masked count."""
    from mimeo_b200 import tandem
    from mimeo_b200.genome import Genome
    prm = dict(to.DEFAULTS, **p)
    m, runs = tandem.record_masks(seqs, prm, runs=True)
    for k, s in enumerate(seqs):
        want = to.mask(s, **prm) if len(s) else (0, [])
        assert (int(m[k]), runs[k]) == want, f'record {k} (L {len(s)}) {prm}: gpu {int(m[k])} {runs[k][:5]} != oracle {want[0]} {want[1][:5]}'
    m2, none = tandem.record_masks(seqs, prm)
    assert none is None and (m2 == m).all()
    idx = [k for k, s in enumerate(seqs) if len(s)]
    g = Genome([str(k) for k in idx], [np.frombuffer(seqs[k], np.uint8) for k in idx])
    try:
        spans = (np.arange(len(idx)), np.zeros(len(idx), np.int64), np.array([len(seqs[k]) for k in idx], np.int64))
        hm, hruns = tandem.masked_runs(g, *spans, prm)
        assert (hm == m[idx]).all() and hruns == [runs[k] for k in idx]
        assert (tandem.masked_counts(g, *spans, prm) == m[idx]).all()
    finally:
        g.close()
    return int(m.sum())


@pytest.mark.parametrize('P', [1, 50, 64, 65, 128, 129, 256])
def test_records_match_oracle_at_every_layout(P):
    rng = np.random.default_rng(1000 + P)
    periods = sorted({1, 2, max(1, P // 2), max(1, P - 1), P} | set(rng.integers(1, P + 1, 6).tolist()))
    seqs = []
    for k, d in enumerate(periods):
        s = planted(rng, int(rng.integers(2 * P + 100, 4 * P + 400)), d, max(3.0, 150 / d), sub=float(rng.choice([0, 0.03])),
                    lower=k % 3 == 1, ns=k % 3)
        seqs.append(n_run(rng, s, int(rng.integers(3, 12))) if k % 2 else s)
    seqs += [random_seq(rng, 700), b'', b'A', b'AC', b'nN', seqs[0]]            # duplicate sequence as a separate record
    assert check_records(seqs, maxperiod=P) > 0


def test_non_default_scores():
    rng = np.random.default_rng(12)
    seqs = [planted(rng, 900, int(rng.integers(1, 30)), 20, sub=0.05, lower=k % 2 == 0, ns=k % 4) for k in range(10)]
    assert check_records(seqs, match=3, mismatch=4, delta=2, minscore=30, maxperiod=33) > 0


def test_16_bit_storage_over_several_batches():
    """minscore + mismatch > 255 stores 16-bit scores; at P = 256 that is 512 bytes per base, so three 400 kbp records
    need two launches under the default 512 MiB storage bound."""
    from mimeo_b200 import _lib, tandem
    from mimeo_b200.genome import Genome
    rng = np.random.default_rng(13)
    seqs = []
    for _ in range(3):
        big = bytearray(random_seq(rng, 400_000))
        for at in range(2000, 395_000, 23_000):
            arr = planted(rng, 0, int(rng.integers(1, 257)), float(rng.uniform(3, 12)), sub=0.02, lower=rng.random() < 0.3)
            arr = n_run(rng, arr, 4) if rng.random() < 0.3 else arr
            big[at:at + len(arr)] = arr
        seqs.append(bytes(big[:400_000]))
    seqs.append(planted(rng, 3000, 200, 6, sub=0.01))
    prm = dict(to.DEFAULTS, minscore=300, mismatch=7, maxperiod=256)
    assert check_records(seqs, **{k: prm[k] for k in ('minscore', 'mismatch', 'maxperiod')}) > 0
    g = Genome([str(k) for k in range(len(seqs))], [np.frombuffer(s, np.uint8) for s in seqs])
    try:
        before = _lib.launch_count()
        tandem.masked_counts(g, np.arange(len(seqs)), np.zeros(len(seqs)), np.array([len(s) for s in seqs]), prm)
        assert _lib.launch_count() - before == 2
    finally:
        g.close()


def test_refusals():
    from mimeo_b200 import _lib, tandem
    seqs = [b'ACGT' * 100, b'']
    for bad in (dict(maxperiod=257), dict(maxperiod=0), dict(match=0), dict(minscore=65530, mismatch=7), dict(delta=-1),
                dict(match=10_000_000)):
        with pytest.raises(_lib.Mb2Error) as e:
            tandem.record_masks(seqs, dict(to.DEFAULTS, **bad), runs=True)
        assert e.value.code == -2
    assert 'overflows the 32-bit scores' in str(e.value)


def test_filter_cli_on_gpu_matches_oracle(tmp_path, monkeypatch):
    text = fasta_text(library())
    kept, masked = check_outputs(tmp_path, monkeypatch, text, [], 40.0)
    assert 0 < kept.count('>') < masked.count('>')
    p = dict(match=3, mismatch=4, delta=2, minscore=30, maxperiod=80)
    check_outputs(tmp_path, monkeypatch, fasta_text(library(8), eol=b'\n'),
                  ['--tmatch', '3', '--tmismatch', '4', '--tdelta', '2', '--tminscore', '30', '--tmaxperiod', '80', '--maxtandem', '25'],
                  25.0, p, outdir='o2', outfile='lib.fa')


def test_filter_cli_reports_score_overflow(tmp_path, monkeypatch, capsys):
    (tmp_path / 'lib.fa').write_bytes(b'>a\n' + b'ACGT' * 75 + b'\n')
    assert run_cli(monkeypatch, ['filter', '--infile', str(tmp_path / 'lib.fa'), '-d', str(tmp_path), '--tmatch', '10000000']) == 1
    out = capsys.readouterr().out
    assert "Error running command 'filter'" in out and 'overflows the 32-bit scores' in out
