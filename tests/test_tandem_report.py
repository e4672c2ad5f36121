"""The tandem-repeat report of `--reportTRF` (DESIGN §2, R1-R6) on CPU: the C oracle (tests/tandem_report_oracle.c) against an
independent numpy statement and the known answers; the kernel source (mimeo_b200/csrc/tandem_report_warp.cuh) on the warp
emulator against the oracle; and both CLIs with the device call stubbed by the oracles, against the oracle pipelines of
tests/tandem_report_reference.py. GPU twin: test_gpu_tandem_report.py."""
import ctypes as C
import math
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import lastz_oracle as lo
from oracle import tandem_oracle as to
from tests import tandem_report_reference as trr
from tests.test_filter_cli import fasta_text, library
from tests.test_tandem_emu import _CODE, planted, random_seq

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SO = os.path.join(HERE, 'emu', '_build', 'libtandem_report_emu.so')
SRCS = [os.path.join(HERE, 'emu', 'tandem_report_emu.cpp'), os.path.join(HERE, 'emu', 'ydrop_emu.h'),
        os.path.join(ROOT, 'mimeo_b200', 'csrc', 'tandem_report_warp.cuh')]


# ---------------------------------------------------------------- an independent statement of R1-R6
def statement(run, M=2, X=7, P=50):
    u = np.frombuffer(bytes(run).upper(), np.uint8)
    code = np.full(256, -1, np.int64)
    for k, b in enumerate(b'ACGT'):
        code[b] = k
    b = code[u]
    L = len(u)
    D = min(P, L - 1)
    c = np.array([int(((b[:L - d] >= 0) & (b[:L - d] == b[d:])).sum()) for d in range(1, D + 1)], np.int64)
    p = int(np.flatnonzero(10 * c >= 9 * c.max())[0]) + 1
    n = np.zeros((p, 4), np.int64)
    ok = b >= 0
    np.add.at(n, (np.arange(L)[ok] % p, b[ok]), 1)
    cons = ''.join('N' if n[k].max() == 0 else 'ACGT'[int(np.argmax(n[k]))] for k in range(p))
    cc = np.array([cons[x % p] for x in range(L)])
    matches = int(sum(1 for x in range(L) if ok[x] and 'ACGT'[b[x]] == cc[x]))
    cp = int(c[p - 1])
    return p, M * cp - X * (L - p - cp), matches, tuple(int(v) for v in n.sum(0)), cons


def runs_for(rng, P, count):
    out = []
    for _ in range(count):
        kind = int(rng.integers(0, 4))
        n = int(rng.integers(2, 3 * P + 80))
        if kind == 0:
            out.append(random_seq(rng, n, b'ACGTNacgtRYKM' if rng.random() < 0.4 else b'ACGT'))
        else:
            period = int(rng.integers(1, P + 1))
            s = planted(rng, 0, period, float(rng.uniform(1.2, 10)), sub=float(rng.choice([0, 0.03, 0.15])),
                        lower=bool(rng.random() < 0.3), ns=int(rng.integers(0, 4)))
            out.append(s if len(s) >= 2 else s + b'A')
    return out


@pytest.mark.parametrize('P', [1, 7, 50, 256])
def test_oracle_matches_independent_statement(P):
    rng = np.random.default_rng(300 + P)
    runs = runs_for(rng, P, 60) + [b'AC', b'nN', b'acgtRYacgt', b'N' * 9, b'ACGTACGTAC'[:P + 1] if P < 9 else b'ACG' * 3]
    for run in runs:
        M, X = int(rng.integers(1, 5)), int(rng.integers(0, 12))
        assert trr.report(run, M, X, P) == statement(run, M, X, P), (run[:40], M, X, P)


KNOWN = [  # run, period, copies, consensus, matches, pmatch, counts, score, entropy
    (b'AT' * 30, 2, '30.0', 'AT', 60, 100, (30, 0, 0, 30), 116, '1.00'),
    (b'A' * 40, 1, '40.0', 'A', 40, 100, (40, 0, 0, 0), 78, '0.00'),
    (b'ACGACGACNACG', 3, '4.0', 'ACG', 11, 91, (4, 4, 3, 0), 0, '1.57'),
    (b'acgtACGTacgaACGT', 4, '4.0', 'ACGT', 15, 93, (5, 4, 4, 3), 6, '1.98'),
    (b'AAGAAGAGAAGAAG', 3, '4.7', 'AGA', 10, 71, (9, 0, 5, 0), 4, '0.94'),
    (b'AGAGTCAGTCAGTC', 4, '3.5', 'TCAG', 12, 85, (4, 3, 4, 3), 2, '1.99'),
]


@pytest.mark.parametrize('case', KNOWN, ids=[k[0][:12].decode() for k in KNOWN])
def test_known_answers(case):
    from mimeo_b200 import tandem
    run, p, copies, cons, matches, pmatch, counts, score, ent = case
    assert trr.report(run, 2, 7, 50) == (p, score, matches, counts, cons) == statement(run, 2, 7, 50)
    row = tandem.report_row('s', 11, 10 + len(run), 7, tandem.Repeat(0, len(run) - 1, p, score, matches, counts, cons))
    comp = ','.join(f'{b}:{100 * c // len(run)}' for b, c in zip('ACGT', counts))
    assert row == (f's\tmimeo-trf\ttandem_repeat\t11\t{10 + len(run)}\t{score}\t+\t.\tID=TR_00007;period={p};copies={copies};'
                   f'consensus={cons};pmatch={pmatch};composition={comp};entropy={ent}\n')
    assert row == trr.gff_row('s', 11, 10 + len(run), 7, (p, score, matches, counts, cons))


def test_entropy_has_no_negative_zero():
    from mimeo_b200 import tandem
    assert tandem.report_row('s', 1, 5, 1, tandem.Repeat(0, 4, 1, 0, 0, (0, 0, 0, 0), 'N')).endswith(';entropy=0.00\n')
    assert tandem.report_row('s', 1, 5, 1, tandem.Repeat(0, 4, 1, 0, 5, (0, 0, 5, 0), 'G')).endswith(';entropy=0.00\n')
    assert math.isclose(float(tandem.report_row('s', 1, 4, 1, tandem.Repeat(0, 3, 1, 0, 1, (1, 1, 1, 1), 'A')).split('entropy=')[1]), 2.0)


# ---------------------------------------------------------------- the kernel source on the warp emulator
def build(so, flags):
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in SRCS):
        os.makedirs(os.path.dirname(so), exist_ok=True)
        tmp = f'{so}.{os.getpid()}.tmp'
        subprocess.check_call(['g++'] + flags + ['-std=c++17', '-shared', '-fPIC', '-I', os.path.join(HERE, 'emu'), '-o', tmp, SRCS[0]])
        os.replace(tmp, so)
    l = C.CDLL(so)
    l.emu_tandem_report.restype = None
    l.emu_tandem_report.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_char_p]
    return l


def shifts_for(P):
    """Shifts per lane the library picks for a maximum period (tandem.cu: 1 up to 32, 2 up to 64, 4 up to 128, 8 up to 256)."""
    return 1 if P <= 32 else 2 if P <= 64 else 4 if P <= 128 else 8


def emu_report(l, run, M=2, X=7, P=50, NT=None):
    s = np.ascontiguousarray(_CODE[np.frombuffer(run, np.uint8)])
    out = np.zeros(7, np.int64)
    cons = C.create_string_buffer(P)
    l.emu_tandem_report(s.ctypes.data, len(s), M, X, P, NT or shifts_for(P), out.ctypes.data, cons)
    p = int(out[0])
    return p, int(out[1]), int(out[2]), tuple(int(v) for v in out[3:7]), cons.raw[:p].decode()


def check_emu(l, run, M=2, X=7, P=50, NT=None):
    want = trr.report(run, M, X, P)
    got = emu_report(l, run, M, X, P, NT)
    assert got == want, f'emulated kernel {got} != oracle {want} (L {len(run)}, M {M}, X {X}, P {P}, NT {NT})'
    return want[0]


def test_kernel_source_planted_periods_1_to_256():
    l = build(SO, ['-O2'])
    rng = np.random.default_rng(41)
    found = 0
    for period in range(1, 257):
        run = planted(rng, 0, period, float(rng.uniform(2.2, 5)) + 8 / period, sub=float(rng.choice([0, 0.02])), lower=period % 5 == 0,
                      ns=period % 3)
        found += check_emu(l, run, P=256) == period
    assert found > 200                                     # R2 recovers most planted periods


@pytest.mark.parametrize('seed', range(4))
def test_kernel_source_random_runs_every_shift_count(seed):
    l = build(SO, ['-O2'])
    rng = np.random.default_rng(700 + seed)
    for P in (1, 7, 31, 32, 33, 50, 64, 65, 100, 128, 129, 200, 256):
        for run in runs_for(rng, P, 4):
            check_emu(l, run, int(rng.integers(1, 5)), int(rng.integers(0, 12)), P)
    run = planted(rng, 0, 20, 9, sub=0.05)
    for NT in (1, 2, 4, 8):                                # more shifts per lane than P needs changes nothing
        check_emu(l, run, P=32, NT=NT)


def test_kernel_source_runs_over_several_tiles():
    """A tile is 64 words of 32 bases; these runs span up to five tiles, with periods below and above 32."""
    l = build(SO, ['-O2'])
    rng = np.random.default_rng(42)
    seen = set()
    for period, P in ((1, 50), (2, 7), (13, 50), (31, 64), (32, 64), (33, 100), (47, 50), (97, 128), (200, 256), (256, 256)):
        run = planted(rng, 0, period, 9000 / period, sub=0.03, ns=4)
        seen.add(check_emu(l, run, P=P) < 32)
    check_emu(l, random_seq(rng, 4100), P=256)
    check_emu(l, b'ACGTTGCA' * 300 + b'N' * 2100 + b'acgttgca' * 200, P=20)
    assert seen == {True, False}


ASAN_CHILD = r'''
import sys, numpy as np
sys.path.insert(0, %(root)r)
from tests import test_tandem_report as T
l = T.build(%(so)r, ['-O1', '-g', '-fsanitize=address', '-fno-omit-frame-pointer'])
rng = np.random.default_rng(902)
for P in (1, 9, 32, 50, 64, 100, 256):
    for run in T.runs_for(rng, P, 5) + [T.planted(rng, 0, min(P, 40), 3000 / min(P, 40), sub=0.03)]:
        T.check_emu(l, run, P=P, X=int(rng.integers(0, 9)))
print('ASAN-SWEEP-OK')
'''


def test_kernel_source_under_address_sanitizer():
    """Bounds of the kernel source (staged words, phase counters, sequence reads, outputs) with the emulator built
    -fsanitize=address."""
    asan = subprocess.run(['g++', '-print-file-name=libasan.so'], capture_output=True, text=True).stdout.strip()
    if not asan or not os.path.isabs(asan) or not os.path.exists(asan):
        pytest.skip('libasan not installed')
    so = os.path.join(HERE, 'emu', '_build', 'libtandem_report_emu_asan.so')
    env = dict(os.environ, LD_PRELOAD=asan, ASAN_OPTIONS='detect_leaks=0:abort_on_error=0')
    r = subprocess.run([sys.executable, '-c', ASAN_CHILD % dict(root=ROOT, so=so)], env=env, capture_output=True, text=True, timeout=900)
    assert 'ERROR: AddressSanitizer' not in r.stderr, r.stderr[-3000:]
    assert r.returncode == 0 and 'ASAN-SWEEP-OK' in r.stdout, (r.stdout[-500:], r.stderr[-2000:])


# ---------------------------------------------------------------- the CLIs with the device call stubbed by the oracles
def stub_reports(monkeypatch):
    from mimeo_b200 import tandem

    def oracle_reports(genome, scaf, start0, length, p):
        m, reps = [], []
        for c, s, n in zip(np.asarray(scaf).tolist(), np.asarray(start0).tolist(), np.asarray(length).tolist()):
            span = to._ascii(genome[c])[int(s):int(s) + int(n)]
            mm, runs = to.mask(span, **p)
            m.append(mm)
            reps.append([tandem.Repeat(a, e, *trr.report(span[a:e + 1], **p)) for a, e in runs])
        return np.array(m, np.uint64), reps
    monkeypatch.setattr(tandem, 'masked_reports', oracle_reports)


def files(d):
    return {p.name: p.read_bytes() for p in d.iterdir() if p.is_file()}


def run_filter(monkeypatch, tmp_path, text, args, outdir):
    from tests.test_filter_cli import run_cli
    (tmp_path / 'lib.fa').write_bytes(text)
    d = tmp_path / outdir
    assert run_cli(monkeypatch, ['filter', '--infile', str(tmp_path / 'lib.fa'), '-d', str(d)] + args) == 0
    return d


@pytest.mark.parametrize('write_trf', [False, True])
def test_filter_report_matches_oracle_pipeline(tmp_path, monkeypatch, write_trf):
    from tests.test_filter_cli import stub_mask
    stub_mask(monkeypatch)
    stub_reports(monkeypatch)
    text = fasta_text(library())
    p = dict(match=3, mismatch=4, delta=2, minscore=30, maxperiod=33)
    args = ['--outfile', 'lib.fasta', '--tmatch', '3', '--tmismatch', '4', '--tdelta', '2', '--tminscore', '30', '--tmaxperiod', '33']
    args += ['--writeTRF'] if write_trf else []
    plain = files(run_filter(monkeypatch, tmp_path, text, args, 'plain'))
    d = run_filter(monkeypatch, tmp_path, text, args + ['--reportTRF'], 'rep')
    got = files(d)
    want = trr.fasta_text_report(text.decode(), p)
    assert got.pop('lib_TRF.gff3').decode() == want
    assert got == plain                                    # every other output unchanged
    assert want.count('\n') > 12 and '\tsat0\t' not in want and 'sat0\t' in want
    assert set(plain) == ({'lib.fasta', 'lib_TRFmasked.fa'} if write_trf else {'lib.fasta'})


def test_filter_report_without_runs_is_header_only(tmp_path, monkeypatch):
    stub_reports(monkeypatch)
    rng = np.random.default_rng(3)
    text = b'>a\n' + random_seq(rng, 300) + b'\n>b\n\n>c\nAC\n'
    d = run_filter(monkeypatch, tmp_path, text, ['--outfile', 'x.fna', '--reportTRF'], 'o')
    assert (d / 'x_TRF.gff3').read_text() == trr.HEADER
    assert (d / 'x.fna').read_bytes().count(b'>') == 3


def map_setup(tmp_path, monkeypatch):
    from tests.test_host_api import _oracle_device_stubs, _write_genome
    from tests.test_tandem_cli import map_inputs, stub_mask
    _oracle_device_stubs(monkeypatch)
    stub_mask(monkeypatch)
    stub_reports(monkeypatch)
    a, b = map_inputs()
    monkeypatch.chdir(tmp_path)
    _write_genome(tmp_path / 'a.fa', a)
    _write_genome(tmp_path / 'b.fa', b)
    return a, b


def test_map_report_matches_oracle_pipeline(tmp_path, monkeypatch):
    from tests.test_tandem_cli import run_cli
    a, b = map_setup(tmp_path, monkeypatch)
    base = ['map', '--afasta', 'a.fa', '--bfasta', 'b.fa', '--minIdt', '90', '--outfile', 'm.tab', '--gffout', 'm.gff3', '--maxtandem', '40']
    run_cli(monkeypatch, base + ['--writeTRF'])
    plain = files(tmp_path)
    run_cli(monkeypatch, base + ['-r', '--writeTRF', '--reportTRF'])
    got = files(tmp_path)
    _tab, gff = lo.mimeo_map({k: lo.encode(v) for k, v in a.items()}, {k: lo.encode(v) for k, v in b.items()}, minIdt=90, minLen=100)
    want = trr.map_report(gff, {k: v.tobytes() for k, v in a.items()})
    assert got.pop('m_TRF.gff3').decode() == want
    assert got == plain
    rows = [ln for ln in want.splitlines() if not ln.startswith('#')]
    assert len(rows) >= 2 and all(';hit=BHit_' in r for r in rows)
    assert {r.split('\t')[0] for r in rows} == {'scaf000', 'scaf001'}
    # the row of the 300 bp (AC)n array planted at scaffold 0, positions 2000..2299
    ac = [r for r in rows if r.startswith('scaf000\t') and ';period=2;' in r and ('consensus=AC;' in r or 'consensus=CA;' in r)]
    assert ac and all(int(r.split('\t')[3]) <= 2001 and int(r.split('\t')[4]) >= 2300 for r in ac)


def test_map_report_without_maxtandem_warns_and_writes_nothing(tmp_path, monkeypatch, capsys):
    from tests.test_tandem_cli import run_cli
    map_setup(tmp_path, monkeypatch)
    run_cli(monkeypatch, ['map', '--afasta', 'a.fa', '--bfasta', 'b.fa', '--minIdt', '90', '--outfile', 'w.tab', '--gffout', 'w.gff3',
                          '--reportTRF'])
    assert '--reportTRF works only together with --maxtandem' in capsys.readouterr().err
    assert not list(tmp_path.glob('*_TRF.gff3')) and (tmp_path / 'w.gff3').exists()
