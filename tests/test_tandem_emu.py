"""The tandem-mask kernel SOURCE (mimeo_b200/csrc/tandem_warp.cuh: backward pass with clamped storage, forward pass with
the pair test, in-warp merge of the masked runs) executed on the CPU by the 32-lane warp emulator (tests/emu/) and held
to the C oracle (oracle/tandem_oracle.c) span by span: masked count and every merged run. No GPU needed."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import tandem_oracle as to

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SO = os.path.join(HERE, 'emu', '_build', 'libtandem_emu.so')
SRCS = [os.path.join(HERE, 'emu', 'tandem_emu.cpp'), os.path.join(HERE, 'emu', 'ydrop_emu.h'),
        os.path.join(ROOT, 'mimeo_b200', 'csrc', 'tandem_warp.cuh')]
_CODE = np.full(256, 8, dtype=np.uint8)
for _c, _v in zip('ACGT', (0, 5, 6, 3)):
    _CODE[ord(_c)] = _CODE[ord(_c.lower())] = _v


def build(so, flags):
    if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in SRCS):
        os.makedirs(os.path.dirname(so), exist_ok=True)
        subprocess.check_call(['g++'] + flags + ['-std=c++17', '-shared', '-fPIC', '-I', os.path.join(HERE, 'emu'), '-o', so, SRCS[0]])
    l = C.CDLL(so)
    l.emu_tandem.restype = C.c_long
    l.emu_tandem.argtypes = [C.c_void_p, C.c_int] + [C.c_int] * 7 + [C.c_void_p, C.c_void_p, C.c_uint, C.POINTER(C.c_uint)]
    return l


def emu_lib():
    return build(SO, ['-O2'])


def layout_for(P):
    """Diagonals per lane the library picks for a maximum period (tandem.cu: 2 up to 64, 4 up to 128, 8 up to 256)."""
    return 2 if P <= 64 else 4 if P <= 128 else 8


def emu_mask(l, seq, M=2, X=7, G=7, T=50, P=50, K=None, wide=None):
    s = np.ascontiguousarray(_CODE[np.frombuffer(seq, np.uint8) if isinstance(seq, bytes) else np.asarray(seq, np.uint8)])
    K = K or layout_for(P)
    wide = (T + X > 255) if wide is None else wide
    cap = len(s) // 2 + 2
    st, en, k = np.zeros(cap, np.int64), np.zeros(cap, np.int64), C.c_uint(0)
    m = l.emu_tandem(s.ctypes.data, len(s), M, X, G, T, P, K, int(wide), st.ctypes.data, en.ctypes.data, cap, C.byref(k))
    return int(m), list(zip(st[:k.value].tolist(), en[:k.value].tolist()))


def random_seq(rng, n, alphabet=b'ACGT'):
    return bytes(rng.choice(np.frombuffer(alphabet, np.uint8), n).tolist())


def planted(rng, n, period, copies, sub=0.0, lower=False, ns=0):
    """A random span with an array of `copies` copies of a random unit of `period` bases planted in it, point substitutions
    at rate `sub`, optionally soft-masked and with `ns` N bases sprinkled over the array."""
    unit = random_seq(rng, period)
    arr = bytearray((unit * (int(copies) + 1))[:max(1, int(period * copies))])
    for x in range(len(arr)):
        if rng.random() < sub:
            arr[x] = int(rng.choice(np.frombuffer(b'ACGT', np.uint8)))
    for _ in range(ns):
        arr[int(rng.integers(0, len(arr)))] = ord('N')
    if lower:
        arr = bytearray(bytes(arr).lower())
    base = bytearray(random_seq(rng, n))
    at = int(rng.integers(0, max(1, n - len(arr))))
    base[at:at + len(arr)] = arr
    return bytes(base[:max(n, len(arr))])


def check(l, seq, **p):
    want = to.mask(seq, match=p.get('M', 2), mismatch=p.get('X', 7), delta=p.get('G', 7), minscore=p.get('T', 50),
                   maxperiod=p.get('P', 50))
    got = emu_mask(l, seq, **p)
    assert got == want, f'emulated kernel {got[0]} {got[1][:6]} != oracle {want[0]} {want[1][:6]} (n {len(seq)}, {p})'
    return want[0]


@pytest.mark.parametrize('seed', range(6))
def test_kernel_source_matches_oracle_random_and_planted(seed):
    l = emu_lib()
    rng = np.random.default_rng(500 + seed)
    masked = 0
    for _ in range(40):
        P = int(rng.choice([1, 2, 7, 13, 31, 50, 64]))
        period = int(rng.integers(1, P + 1))
        n = int(rng.integers(0, 400))
        kind = int(rng.integers(0, 4))
        if kind == 0:
            seq = random_seq(rng, n, b'ACGTNacgtRY' if rng.random() < 0.3 else b'ACGT')
        else:
            seq = planted(rng, n, period, float(rng.uniform(1.5, 12)), sub=float(rng.choice([0, 0.03, 0.1])),
                          lower=bool(rng.random() < 0.3), ns=int(rng.integers(0, 3)))
        M, X, G = int(rng.integers(1, 5)), int(rng.integers(0, 12)), int(rng.integers(0, 12))
        T = int(rng.integers(1, 80))
        masked += check(l, seq, M=M, X=X, G=G, T=T, P=P)
    assert masked > 0


def test_kernel_source_every_layout_and_storage_width():
    l = emu_lib()
    rng = np.random.default_rng(77)
    for P, K in ((50, 2), (50, 4), (50, 8), (100, 4), (100, 8), (200, 8), (256, 8)):
        for wide in (False, True):
            for period in (1, P // 3 + 1, P):
                seq = planted(rng, 3 * P + 50, period, max(2.0, 160 / period + 1), sub=0.02)
                check(l, seq, P=P, K=K, wide=wide)
    # T + X beyond one byte: 16-bit storage
    seq = planted(rng, 700, 4, 150)
    check(l, seq, T=300, X=9, P=20, wide=True)


def test_kernel_source_long_span_and_edges():
    l = emu_lib()
    rng = np.random.default_rng(78)
    seq = planted(rng, 6000, 37, 40, sub=0.05) + b'(AC)' + random_seq(rng, 100)
    check(l, seq)
    for n in (0, 1, 2, 3, 4):
        check(l, b'A' * n, T=1)
    check(l, b'AC' * 40)
    check(l, b'ac' * 40)


ASAN_CHILD = r'''
import sys, numpy as np
sys.path.insert(0, %(root)r)
from tests import test_tandem_emu as T
l = T.build(%(so)r, ['-O1', '-g', '-fsanitize=address', '-fno-omit-frame-pointer'])
rng = np.random.default_rng(901)
for k in range(30):
    P = int(rng.choice([1, 9, 50, 64, 100, 256]))
    seq = T.planted(rng, int(rng.integers(0, 900)), int(rng.integers(1, P + 1)), float(rng.uniform(1, 8)), sub=0.03, ns=1)
    T.check(l, seq, P=P, T=int(rng.integers(10, 300)), X=int(rng.integers(0, 9)))
print('ASAN-SWEEP-OK')
'''


def test_kernel_source_under_address_sanitizer():
    """Bounds of the kernel source (stored anti-diagonals, ring, sequence reads) with the emulator built -fsanitize=address."""
    import sys
    asan = subprocess.run(['g++', '-print-file-name=libasan.so'], capture_output=True, text=True).stdout.strip()
    if not asan or not os.path.isabs(asan) or not os.path.exists(asan):
        pytest.skip('libasan not installed')
    so = os.path.join(HERE, 'emu', '_build', 'libtandem_emu_asan.so')
    env = dict(os.environ, LD_PRELOAD=asan, ASAN_OPTIONS='detect_leaks=0:abort_on_error=0')
    r = subprocess.run([sys.executable, '-c', ASAN_CHILD % dict(root=ROOT, so=so)], env=env, capture_output=True, text=True, timeout=900)
    assert 'ERROR: AddressSanitizer' not in r.stderr, r.stderr[-3000:]
    assert r.returncode == 0 and 'ASAN-SWEEP-OK' in r.stdout, (r.stdout[-500:], r.stderr[-2000:])
