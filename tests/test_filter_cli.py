"""`mimeo filter [--writeTRF]` on CPU: the product's host path (CLI, native FASTA reader, keep/drop rule, N replacement,
FASTA writer, output paths) with the mask stubbed by its oracle, against filter_reference.fasta_filter. GPU twin:
test_gpu_filter.py."""
import sys

import numpy as np
import pytest

from oracle import tandem_oracle as to
from tests import filter_reference as fr
from tests.test_tandem_emu import planted, random_seq


def library(seed=71):
    """(header, sequence) records: planted arrays of periods 1-50 (some soft-masked, some broken by N), random records, lower
    case and IUPAC bytes, duplicate ids, multi-word headers, and records of length 0, 1 and 2."""
    rng = np.random.default_rng(seed)
    recs = []
    for k, period in enumerate((1, 2, 3, 4, 6, 9, 13, 21, 34, 50)):
        seq = planted(rng, int(rng.integers(120, 1500)), period, float(rng.uniform(3, 12)) + 100 / period,
                      sub=float(rng.choice([0, 0.03])), lower=k % 3 == 0, ns=3 * (k % 2))
        recs.append((f'sat{k} period={period} planted array', seq))
    for k in range(6):
        recs.append((f'plain{k}', random_seq(rng, int(rng.integers(60, 900)))))
    recs.append(('iupac mixed case', random_seq(rng, 400, b'ACGTacgtRYKMSWBDHVNnrykm')))
    recs.append(('iupac_array', b'ACGT' * 10 + b'acRYacRYacRYacRYacRYacRYacRYacRYacRYacRYacRY' * 3 + b'TTGCA' * 8))
    recs.append(('dup first copy', b'AC' * 70))
    recs.append(('dup second copy', random_seq(rng, 300)))
    recs.append(('empty record', b''))
    recs.append(('one', b'A'))
    recs.append(('two', b'AA'))
    recs.append(('twoN', b'nN'))
    return recs


def fasta_text(recs, eol=b'\r\n', width=70):
    """A FASTA file of the records with `eol` line ends, lines of `width` bases and a blank line after every third record."""
    out = [b'; a comment before the first record' + eol]
    for k, (h, s) in enumerate(recs):
        out.append(b'>' + h.encode() + eol)
        out += [s[i:i + width] + eol for i in range(0, len(s), width)]
        if k % 3 == 2:
            out.append(eol)
    return b''.join(out)


def stub_mask(monkeypatch):
    from mimeo_b200 import tandem

    def oracle_masks(seqs, p, runs=False):
        res = [to.mask(s, **p) if len(s) else (0, []) for s in seqs]
        return np.array([r[0] for r in res], np.uint64), ([r[1] for r in res] if runs else None)
    monkeypatch.setattr(tandem, 'record_masks', oracle_masks)


def run_cli(monkeypatch, argv):
    from mimeo_b200 import app
    monkeypatch.setattr(sys, 'argv', ['mimeo'] + argv)
    try:
        app.main()
    except SystemExit as e:
        return e.code or 0
    return 0


def check_outputs(tmp_path, monkeypatch, text, args, maxtandem, params=None, outdir='out/sub', outfile='lib.fasta'):
    """Runs `mimeo filter` with and without --writeTRF and compares both files with filter_reference, byte for byte."""
    (tmp_path / 'lib.fa').write_bytes(text)
    base = ['filter', '--infile', str(tmp_path / 'lib.fa'), '-d', str(tmp_path / outdir), '--outfile', outfile] + args
    want_kept, want_masked = fr.fasta_filter(text.decode(), maxtandem, params)
    stem = outfile.rsplit('.', 1)[0] if outfile.endswith(('.fa', '.fasta', '.fna')) else outfile
    masked = tmp_path / outdir / (stem + '_TRFmasked.fa')
    masked.unlink(missing_ok=True)
    assert run_cli(monkeypatch, base) == 0
    assert (tmp_path / outdir / outfile).read_bytes() == want_kept.encode()
    assert not masked.exists()
    assert run_cli(monkeypatch, base + ['--writeTRF']) == 0
    assert (tmp_path / outdir / outfile).read_bytes() == want_kept.encode()
    assert masked.read_bytes() == want_masked.encode()
    return want_kept, want_masked


@pytest.mark.parametrize('maxtandem', [None, '0', '12.5', '100'])
def test_filter_matches_oracle(tmp_path, monkeypatch, maxtandem):
    stub_mask(monkeypatch)
    recs = library()
    args = [] if maxtandem is None else ['--maxtandem', maxtandem]
    mt = 40.0 if maxtandem is None else float(maxtandem)
    kept, masked = check_outputs(tmp_path, monkeypatch, fasta_text(recs), args, mt)
    n_kept = kept.count('>')
    if mt == 100:
        assert n_kept == len(recs)
    else:
        assert 0 < n_kept < len(recs)                                       # some records dropped, some kept
    assert '>empty record\n>one\nA\n>two\n' in kept                           # L = 0, 1 and 2 are kept
    assert '\n>dup first copy\n' in masked and '\n>dup second copy\n' in masked
    body = ''.join(ln for ln in masked.splitlines() if not ln.startswith('>'))
    assert set('RYKMSWBDHVacgtrykm') <= set(body)                           # case and IUPAC bytes preserved
    assert masked.count('N') > text_count(recs, b'N') + text_count(recs, b'n')   # some positions were masked


def text_count(recs, c):
    return sum(s.count(c) for _h, s in recs)


def test_filter_lf_files_output_paths_and_ignored_flags(tmp_path, monkeypatch):
    stub_mask(monkeypatch)
    text = fasta_text(library(5), eol=b'\n', width=60)
    check_outputs(tmp_path, monkeypatch, text, ['--TRFpath', '/no/such/trf', '--tPM', '1', '--tPI', '99'], 40.0, outdir='.',
                  outfile='segments.fna')
    check_outputs(tmp_path, monkeypatch, text, [], 40.0, outdir='o', outfile='library')


def test_filter_non_default_mask_parameters(tmp_path, monkeypatch):
    stub_mask(monkeypatch)
    p = dict(match=3, mismatch=4, delta=2, minscore=30, maxperiod=33)
    args = ['--tmatch', '3', '--tmismatch', '4', '--tdelta', '2', '--tminscore', '30', '--tmaxperiod', '33', '--maxtandem', '25']
    check_outputs(tmp_path, monkeypatch, fasta_text(library(8)), args, 25.0, p)


def test_record_masked_exactly_maxtandem_percent_is_kept(tmp_path, monkeypatch):
    stub_mask(monkeypatch)
    recs = library()
    h, s = recs[3]
    m, _ = to.mask(s)
    assert 0 < m < len(s)
    at = 100.0 * m / len(s)
    kept, _ = check_outputs(tmp_path, monkeypatch, fasta_text(recs), ['--maxtandem', repr(at)], at)
    assert '>' + h + '\n' in kept
    below = float(np.nextafter(at, 0.0))
    kept, _ = check_outputs(tmp_path, monkeypatch, fasta_text(recs), ['--maxtandem', repr(below)], below)
    assert '>' + h + '\n' not in kept


def test_every_record_dropped_writes_empty_outfile(tmp_path, monkeypatch, capsys):
    stub_mask(monkeypatch)
    recs = library()[:10]                                                      # planted arrays only
    (tmp_path / 'lib.fa').write_bytes(fasta_text(recs))
    out = tmp_path / 'kept.fa'
    assert run_cli(monkeypatch, ['filter', '--infile', str(tmp_path / 'lib.fa'), '-d', str(tmp_path), '--outfile', 'kept.fa',
                                 '--maxtandem', '0', '--tminscore', '4', '--writeTRF']) == 0
    assert out.exists() and out.read_bytes() == b''
    assert (tmp_path / 'kept_TRFmasked.fa').read_bytes() == fr.fasta_filter(fasta_text(recs).decode(), 0.0, dict(minscore=4))[1].encode()
    err = capsys.readouterr().err
    assert 'Every record was removed by the tandem repeat filter' in err and '0 of 10 records kept (maxtandem 0.0%)' in err


@pytest.mark.parametrize('flag,value', [('--tmatch', '0'), ('--tmismatch', '-1'), ('--tdelta', '-2'), ('--tminscore', '0'),
                                        ('--tmaxperiod', '0'), ('--tmaxperiod', '257'), ('--tminscore', '65530'),
                                        ('--maxtandem', '-1'), ('--maxtandem', '101'), ('--maxtandem', 'nan')])
def test_filter_rejects_bad_values(tmp_path, monkeypatch, capsys, flag, value):
    (tmp_path / 'lib.fa').write_bytes(b'>a\nACGT\n')
    assert run_cli(monkeypatch, ['filter', '--infile', str(tmp_path / 'lib.fa'), '-d', str(tmp_path / 'o'), flag, value]) == 1
    out = capsys.readouterr().out
    assert "Error running command 'filter'" in out and flag in out
    assert not (tmp_path / 'o').exists()                                        # refused before anything is written


@pytest.mark.parametrize('case', ['no_flag', 'missing_file', 'empty_file', 'no_records'])
def test_filter_exits_1_without_input_records(tmp_path, monkeypatch, capsys, case):
    argv = ['filter', '-d', str(tmp_path / 'o')]
    if case != 'no_flag':
        argv += ['--infile', str(tmp_path / 'lib.fa')]
    if case == 'empty_file':
        (tmp_path / 'lib.fa').write_bytes(b'')
    if case == 'no_records':
        (tmp_path / 'lib.fa').write_bytes(b'ACGT\nno header line\n')
    assert run_cli(monkeypatch, argv) == 1
    err = capsys.readouterr().err
    assert ('No sequences found' in err) == (case in ('empty_file', 'no_records'))
    assert not (tmp_path / 'o').exists()


def test_usage_lists_filter(monkeypatch, capsys):
    assert run_cli(monkeypatch, []) == 1
    assert '  filter  ' in capsys.readouterr().out


def test_reference_fasta_filter_known_answer():
    """Exact arrays scoring far above T are masked end to end, a 10 bp record cannot reach T = 50 (at most 2 * 9)."""
    text = '>sat a b\r\n' + 'AC' * 40 + '\r\n\r\n>flank\n' + 'ACGTTGCAAG\n>empty\n>sat2\n' + 'ac' * 20 + '\n' + 'ac' * 15 + '\n'
    kept, masked = fr.fasta_filter(text, 40)
    assert kept == '>flank\nACGTTGCAAG\n>empty\n'
    assert masked == '>sat a b\n' + 'N' * 60 + '\n' + 'N' * 20 + '\n>flank\nACGTTGCAAG\n>empty\n>sat2\n' + 'N' * 60 + '\n' + 'N' * 10 + '\n'
    assert fr.fasta_filter(text, 100)[0] == ('>sat a b\n' + 'AC' * 30 + '\n' + 'AC' * 10 + '\n>flank\nACGTTGCAAG\n>empty\n>sat2\n'
                                             + 'ac' * 30 + '\n' + 'ac' * 5 + '\n')
