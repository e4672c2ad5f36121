"""The C oracle of the tandem-repeat mask (oracle/tandem_oracle.c) against an independent pure-Python statement and
known answers (DESIGN §2, T1-T4)."""
import numpy as np
import pytest

from oracle import tandem_oracle as to

NEG = float('-inf')


def _sub(a, b, M, X):
    a, b = a.upper(), b.upper()
    return M if a == b and a in 'ACGT' else -X


def _prefix_best(s, p, q, M, X, G, P):
    """Best local alignment in the strip ending exactly at prefix cell (p, q) (0 on the boundary), by its own DP."""
    if p == 0 or q == 0:
        return 0
    H = [[NEG] * (q + 1) for _ in range(p + 1)]
    for i in range(p + 1):
        for j in range(q + 1):
            if i == 0 or j == 0:
                H[i][j] = 0
            elif 1 <= j - i <= P:
                v = max(0, H[i - 1][j - 1] + _sub(s[i - 1], s[j - 1], M, X))
                v = max(v, H[i - 1][j] - G, H[i][j - 1] - G)
                H[i][j] = v
    return H[p][q]


def python_mask(s, M, X, G, T, P):
    """Masked positions: for each pair (p, q), 1 <= q-p <= P, best = prefix DP ending at (p, q) + sub + suffix DP starting
    at (p+1, q+1), the suffix one computed as a prefix DP of the reversed sequence (strip diagonals are the same there)."""
    n = len(s)
    r = s[::-1]
    mask = [False] * n
    for p in range(n):
        for q in range(p + 1, min(n, p + P + 1)):
            suf = _prefix_best(r, n - q - 1, n - p - 1, M, X, G, P)
            if _prefix_best(s, p, q, M, X, G, P) + _sub(s[p], s[q], M, X) + suf >= T:
                for x in range(p, q + 1):
                    mask[x] = True
    return sum(mask)


@pytest.mark.parametrize('seed', range(4))
def test_oracle_matches_independent_python_statement(seed):
    rng = np.random.default_rng(seed)
    for _ in range(6):
        n = int(rng.integers(0, 33))
        unit = ''.join(rng.choice(list('ACGT'), int(rng.integers(1, 6))))
        s = list((unit * 40)[:n]) if rng.random() < 0.6 else list(rng.choice(list('ACGTN'), n))
        for _k in range(int(rng.integers(0, 4))):
            if n:
                s[int(rng.integers(0, n))] = str(rng.choice(list('ACGTNacgt')))
        s = ''.join(s)
        M, X, G = int(rng.integers(1, 4)), int(rng.integers(0, 8)), int(rng.integers(0, 8))
        T, P = int(rng.integers(1, 30)), int(rng.integers(1, 9))
        want = python_mask(s, M, X, G, T, P)
        got = to.mask(s, M, X, G, T, P)[0]
        assert got == want, (s, M, X, G, T, P)


def _unit_without_self_match(rng, d):
    """A random unit of period d whose array has no self-match on any diagonal but multiples of d that could score."""
    while True:
        u = ''.join(rng.choice(list('ACGT'), d))
        arr = u * 5
        ok = all(sum(arr[x] == arr[x + k] for x in range(len(arr) - k)) < 0.5 * (len(arr) - k) for k in range(1, d))
        if ok and len(set(u)) == 4:
            return u


def test_known_answers():
    assert to.mask('AC' * 40) == (80, [(0, 79)])
    rng = np.random.default_rng(3)
    u = _unit_without_self_match(rng, 10)
    assert to.mask((u * 4)[:35])[0] == 35                 # 2 * (35 - 10) = 50
    assert to.mask((u * 4)[:34])[0] == 0                  # 48
    r60 = ''.join(rng.choice(list('ACGT'), 60))
    assert to.mask(r60 + r60, maxperiod=50)[0] == 0
    assert to.mask(r60 + r60, maxperiod=60)[0] == 120
    arr = 'AC' * 40
    m, iv = to.mask(arr[:40] + 'N' * 60 + arr[:40])      # an N run longer than P: no pair reaches across it
    assert len(iv) == 2 and iv[0][0] == 0 and iv[1][1] == 139 and m < 140
    assert to.mask(arr[:40] + 'N' + arr[41:])[0] == 80        # one N: a mismatch inside the array, which still scores
    assert to.mask(arr.lower()) == to.mask(arr)
    assert to.mask('ACgtAcGt' * 10) == to.mask('ACGT' * 20)
    r10k = ''.join(np.random.default_rng(12345).choice(list('ACGT'), 10_000))
    assert to.mask(r10k)[0] == 0
    assert to.mask('')[0] == 0 and to.mask('A', minscore=1)[0] == 0
