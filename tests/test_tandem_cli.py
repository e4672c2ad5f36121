"""`mimeo map --maxtandem [--writeTRF]` on CPU: the product's host path (CLI, UID order, span gather from the GFF rows,
filtered GFF3, _TRFfiltered.tab) with the alignment and the mask stubbed by their oracles, against the oracle pipeline
(lastz_oracle.mimeo_map followed by tandem_oracle.map_filter). GPU twin: test_gpu_tandem.py."""
import sys

import numpy as np
import pytest

from oracle import lastz_oracle as lo
from oracle import tandem_oracle as to
from tests.helpers import synth_genome
from tests.test_host_api import _oracle_device_stubs, _write_genome


def map_inputs(seed=61):
    """A and B genomes where B carries copies of two A loci (one plain, one holding a microsatellite) and of a
    microsatellite-rich A block, so the filter drops some hits and keeps others."""
    rng = np.random.default_rng(seed)
    a = synth_genome(seed, 2, 9_000, 0)
    b = synth_genome(seed + 1, 2, 7_000, 0)
    a['scaf000'][2000:2300] = np.frombuffer(b'AC' * 150, np.uint8)                  # a 300 bp microsatellite inside a 600 bp locus
    a['scaf001'][1000:1400] = np.frombuffer((b'ACGTT' * 80).lower(), np.uint8)     # soft-masked pentamer array
    for src, at, dst, to_ in (('scaf000', 1800, 'scaf000', 500), ('scaf000', 5000, 'scaf001', 300), ('scaf001', 900, 'scaf001', 3000),
                              ('scaf000', 7000, 'scaf000', 4000)):
        cp = a[src][at:at + 600].copy()
        flip = rng.random(len(cp)) < 0.02
        cp[flip] = np.frombuffer(b'ACGT', np.uint8)[rng.integers(0, 4, int(flip.sum()))]
        b[dst][to_:to_ + 600] = cp
    return a, b


def run_cli(monkeypatch, argv):
    from mimeo_b200 import app
    monkeypatch.setattr(sys, 'argv', ['mimeo'] + argv)
    try:
        app.main()
    except SystemExit as e:
        assert e.code in (0, None)


def stub_mask(monkeypatch):
    from mimeo_b200 import tandem
    monkeypatch.setattr(tandem, 'masked_counts', lambda genome, scaf, start0, length, p: to.masked_counts(genome, scaf, start0, length, p))


def test_map_maxtandem_writetrf_matches_oracle_pipeline(tmp_path, monkeypatch):
    _oracle_device_stubs(monkeypatch)
    stub_mask(monkeypatch)
    a, b = map_inputs()
    monkeypatch.chdir(tmp_path)
    _write_genome(tmp_path / 'a.fa', a)
    _write_genome(tmp_path / 'b.fa', b)
    base = ['map', '--afasta', 'a.fa', '--bfasta', 'b.fa', '--adir', 'A', '--bdir', 'B', '--minIdt', '90']
    run_cli(monkeypatch, base + ['--outfile', 'm.tab', '--gffout', 'm.gff3'])
    tab, gff = lo.mimeo_map({k: lo.encode(v) for k, v in a.items()}, {k: lo.encode(v) for k, v in b.items()}, minIdt=90, minLen=100)
    assert (tmp_path / 'm.gff3').read_text() == gff                                  # without --maxtandem: unchanged
    assert not (tmp_path / 'm_TRFfiltered.tab').exists()
    run_cli(monkeypatch, base + ['-r', '--outfile', 'm.tab', '--gffout', 't.gff3', '--maxtandem', '40', '--writeTRF'])
    want_gff, want_tab = to.map_filter(tab, gff, {k: v.tobytes() for k, v in a.items()}, 40.0, minLen=100, minIdt=90)
    got = (tmp_path / 't.gff3').read_text()
    assert got == want_gff and (tmp_path / 'm_TRFfiltered.tab').read_text() == want_tab
    n_all = sum(1 for ln in gff.splitlines() if not ln.startswith('#'))
    n_kept = sum(1 for ln in got.splitlines() if not ln.startswith('#'))
    assert 0 < n_kept < n_all                                                        # the filter dropped some hits ...
    ids = [int(ln.split('ID=')[1].split(';')[0].rsplit('_', 1)[1]) for ln in got.splitlines() if not ln.startswith('#')]
    assert ids != list(range(1, n_kept + 1))                                         # ... and the survivors keep their UIDs


def test_map_maxtandem_every_row_dropped_writes_headers_only(tmp_path, monkeypatch, capsys):
    _oracle_device_stubs(monkeypatch)
    stub_mask(monkeypatch)
    a, b = map_inputs()
    monkeypatch.chdir(tmp_path)
    _write_genome(tmp_path / 'a.fa', a)
    _write_genome(tmp_path / 'b.fa', b)
    run_cli(monkeypatch, ['map', '--afasta', 'a.fa', '--bfasta', 'b.fa', '--minIdt', '90', '--outfile', 'h.tab', '--gffout', 'h.gff3',
                          '--maxtandem', '0.001', '--tminscore', '2', '--writeTRF'])
    tab, gff = lo.mimeo_map({k: lo.encode(v) for k, v in a.items()}, {k: lo.encode(v) for k, v in b.items()}, minIdt=90, minLen=100)
    assert (tmp_path / 'h.gff3').read_text() == ''.join(ln for ln in gff.splitlines(True) if ln.startswith('#'))
    assert (tmp_path / 'h_TRFfiltered.tab').read_text() == to.map_filter(tab, gff, {k: v.tobytes() for k, v in a.items()}, 0.001,
                                                                          dict(minscore=2), minLen=100, minIdt=90)[1]
    assert 'removed by the tandem repeat filter' in capsys.readouterr().err


@pytest.mark.parametrize('flag,value', [('--tmatch', '0'), ('--tmismatch', '-1'), ('--tdelta', '-2'), ('--tminscore', '0'),
                                        ('--tmaxperiod', '0'), ('--tmaxperiod', '257'), ('--tminscore', '65530')])
def test_map_rejects_bad_tandem_parameters(tmp_path, monkeypatch, capsys, flag, value):
    from mimeo_b200 import app
    monkeypatch.chdir(tmp_path)
    monkeypatch.setattr(sys, 'argv', ['mimeo', 'map', '--afasta', 'a.fa', '--bfasta', 'b.fa', '--maxtandem', '40', flag, value])
    with pytest.raises(SystemExit) as e:
        app.main()
    assert e.value.code == 1
    assert 'Error running command' in capsys.readouterr().out
    assert not any(p.name.startswith('temp_') for p in tmp_path.iterdir())     # refused before any file is written
