"""The merged 4-bit code of the seed scan (mimeo_b200/csrc/seed.cu: nib_merge, s1_entry, s1_prepare, nib_span, nib_rev,
seed_match_merged, xdrop_window30), restated with Python integers and held against the plain per-column statements of
tests/scan_reference.py. No GPU needed.

A genome's nb plane holds 4 bits per base: base | parity << 2 for A, C, G, T (parity = C or G) and 8 for anything else. The
scan merges a target and a query word into m = t ^ q on the base bits and t | q on the parity and non-ACGT bits, and indexes
its first-stage table with three columns of m (12 bits) whose bits 2..3 are xor-ed with bits 8..9."""
import numpy as np
import pytest

from tests import scan_reference as R

M32 = 0xFFFFFFFF
CODES = [0, 5, 6, 3]            # nb code of A, C, G, T
NCODE = 8
DONE = 1 << 24


def nib_code(base, bad):
    return NCODE if bad else base | (((base ^ (base >> 1)) & 1) << 2)


def nib_merge(t, q):
    return ((t ^ q) & 0x33333333) | ((t | q) & 0xCCCCCCCC)


def nib_rev(x):
    return int(''.join(reversed(f'{x:08x}')), 16)


def funnel_r(lo, hi, s):
    return (((hi << 32) | lo) >> (s & 31)) & M32


def column_score(nib):
    """score of one merged column, as s1_entry decodes it"""
    if nib & 8:
        return R.SCORE_N
    t = (nib >> 2) & 1
    return int(R.HOXD70[t, t ^ (nib & 3)])


def s1_entry(idx, X):
    code = idx ^ (((idx >> 8) & 3) << 2)
    p = np.cumsum([column_score((code >> (4 * c)) & 15) for c in range(3)])
    sm, mx, mn = int(p[-1]), int(p.max()), int(p.min())
    return ((sm & 0x3FF) << 22) | ((mx + 125) << 13) | (mn + X + 125)


def s1_prepare(w):
    an = (((w[0] | w[1] | w[2]) & 0x88888888) | (w[3] & 0x00888888)) != 0
    sw = [0x0C00C00C, 0xC00C00C0, 0x00C00C00, 0x0000C00C]
    src = [funnel_r(w[0], w[1], 6), funnel_r(w[1], w[2], 6), funnel_r(w[2], w[3], 6), w[3] >> 6]
    return [w[i] ^ (src[i] & sw[i]) for i in range(4)], an


def s1_bits(w, s):
    if s < 0:
        return (w[0] << -s) & M32
    j, r = s >> 5, s & 31
    return w[j] if r == 0 else (funnel_r(w[j], w[j + 1], r) if j < 3 else w[3] >> r)


def xdrop_window30(tab, w, an, best, D):
    """(best, D, chunks counted) after one prepared window"""
    all10 = an and D < DONE // 2
    parked = 0
    for k in range(10):
        e = tab[(s1_bits(w, 12 * k - 2) & 0x3FFC) >> 2]
        parked += D
        term = (e & 0x1FFF) < D
        dm = max(D, (e >> 13) & 0x1FF)
        best += dm - D
        sm = (e >> 22) - 1024 if e >> 31 else e >> 22
        D = DONE if term else dm - sm
    return best, D, 10 if all10 else 10 - (parked >> 24)


def plane_words(S):
    """the nb plane of a scan_reference Space, 8 codes per word"""
    nib = np.where(S.bad, NCODE, S.base | (((S.base ^ (S.base >> 1)) & 1) << 2)).astype(np.int64)
    nib = np.concatenate([nib, np.full((-len(nib)) % 8 + 16, NCODE, np.int64)])
    return [int(sum(int(v) << (4 * c) for c, v in enumerate(nib[a:a + 8]))) for a in range(0, len(nib), 8)]


def nib_span(words, p, nw):
    w0, sh, odd = (p >> 3) & ~1, (p & 7) * 4, bool(p & 8)
    x = words[w0:w0 + nw + 2]
    return [funnel_r(x[m + 1], x[m + 2], sh) if odd else funnel_r(x[m], x[m + 1], sh) for m in range(nw)]


def span_direct(S, p, n):
    """n columns from p, one code per column"""
    return [nib_code(int(S.base[c]), bool(S.bad[c])) for c in range(p, p + n)]


def words_to_cols(w):
    return [(w[c >> 3] >> (4 * (c & 7))) & 15 for c in range(8 * len(w))]


def test_merged_code_scores_every_pair():
    pairs = [(CODES[a], CODES[b], int(R.HOXD70[a, b])) for a in range(4) for b in range(4)]
    pairs += [(t, q, R.SCORE_N) for t in range(16) for q in range(16) if (t | q) & 8]
    for t, q, want in pairs:
        assert column_score(nib_merge(t, q) & 15) == want, (t, q)
        # the same in every column of a word
        for c in range(8):
            assert column_score((nib_merge(t << (4 * c), q << (4 * c)) >> (4 * c)) & 15) == want


def reachable_column_codes():
    valid = CODES + [NCODE]
    return sorted({nib_merge(t, q) & 15 for t in valid for q in valid})


@pytest.mark.parametrize('X', [251, 910, 6399])
def test_every_table_entry_equals_the_column_rule(X):
    """Every entry of a reachable chunk code: its fields are the prefix sums of the three columns' HOXD70 / SCORE_N scores,
    and one chunk step from any open state equals three column steps."""
    cols = reachable_column_codes()
    assert len(cols) == 10
    rep = {}
    valid = CODES + [NCODE]
    for a, t in enumerate(valid):
        for b, q in enumerate(valid):
            rep.setdefault(nib_merge(t, q) & 15, R.SCORE_N if a == 4 or b == 4 else int(R.HOXD70[a, b]))
    tab = [s1_entry(i, X) for i in range(4096)]
    for c0 in cols:
        for c1 in cols:
            for c2 in cols:
                code = c0 | c1 << 4 | c2 << 8
                idx = code ^ (((code >> 8) & 3) << 2)
                sc = [rep[c0], rep[c1], rep[c2]]
                e = tab[idx]
                for deficit in (0, 1, 50, 250, X - 250, X - 100, X - 1, X):
                    if deficit < 0 or deficit > X:
                        continue
                    # column rule from best = 0, run = -deficit
                    best, run, stop = 0, -deficit, False
                    for s in sc:
                        run += s
                        if run > best:
                            best = run
                        elif run < best - X:
                            stop = True
                            break
                    D = deficit + 125
                    term = (e & 0x1FFF) < D
                    dm = max(D, (e >> 13) & 0x1FF)
                    assert term == stop, (code, deficit)
                    if not stop:
                        sm = (e >> 22) - 1024 if e >> 31 else e >> 22
                        assert dm - D == best and dm - sm - 125 == best - run, (code, deficit)


def test_bank_bits_vary_with_the_target():
    """With the query bases of a chunk fixed, the 64 target triples reach all 32 banks (index bits 0..4)."""
    for qa in range(64):
        banks = set()
        for ta in range(64):
            t = sum(CODES[(ta >> (2 * c)) & 3] << (4 * c) for c in range(3))
            q = sum(CODES[(qa >> (2 * c)) & 3] << (4 * c) for c in range(3))
            w, _ = s1_prepare([nib_merge(t, q), 0, 0, 0])
            banks.add(w[0] & 31)
        assert len(banks) == 32, qa


def test_spans_and_reversal_equal_the_plain_columns():
    rng = np.random.default_rng(7)
    codes = [rng.integers(0, 6, 700).astype(np.uint8)]           # 4, 5: non-ACGT
    S = R.Space(codes)
    words = plane_words(S)
    for p in range(R.END_PAD - 40, R.END_PAD + 760):
        for nw in (4, 8):
            w = nib_span(words, p, nw)
            assert words_to_cols(w) == span_direct(S, p, 8 * nw), (p, nw)
        w = nib_span(words, p, 4)
        assert words_to_cols([nib_rev(w[3 - i]) for i in range(4)]) == span_direct(S, p, 32)[::-1]


def leader_test(tw, qw, i, j, transition):
    """the kernel's leader statement on the merged block of hit (i, j) (nb planes tw, qw; no soft mask): True = not a leader"""
    m = [nib_merge(a, b) for a, b in zip(nib_span(tw, i - 13, 8), nib_span(qw, j - 13, 8))]
    l0, l1, l2 = funnel_r(m[1], m[2], 16), funnel_r(m[2], m[3], 16), m[3] >> 16
    ln = ((l0 | l1) & 0x88888888) | (l2 & 0x888)
    x0, x1, x2 = l0 & 0x30030333, l1 & 0x30303003, l2 & 0x333
    match = (x0 | x1 | x2) == 0 or (bool(transition) and ((x0 | x1 | x2) & 0x11111111) == 0
                                    and bin(x0).count('1') + bin(x1).count('1') + bin(x2).count('1') == 1)
    return ln == 0 and match


def related_pair(seed):
    """a target with N runs and a query that is a diverged copy of it (with other N runs), so that extensions stay open
    through non-ACGT columns and leader windows are often seed hits"""
    rng = np.random.default_rng(seed)
    t = rng.integers(0, 4, 6000).astype(np.uint8)
    q = np.where(rng.random(6000) < 0.12, rng.integers(0, 4, 6000), t).astype(np.uint8)
    for s in (t, q):
        for _ in range(40):
            a = int(rng.integers(0, 5990))
            s[a:a + int(rng.integers(1, 6))] = 4
    return R.Space([t]), R.Space([q])


@pytest.mark.parametrize('transition', [0, 1])
def test_leader_test_on_merged_codes(transition):
    T, Q = related_pair(11)
    tw, qw = plane_words(T), plane_words(Q)
    rng = np.random.default_rng(12)
    n_match = 0
    for _ in range(3000):
        i = int(rng.integers(R.END_PAD + 20, R.END_PAD + 5900))
        j = i + int(rng.integers(-1, 2))
        want = bool(T.seedable[i - 1] and Q.seedable[j - 1] and R.keys_match(T.key[i - 1], Q.key[j - 1], transition))
        assert leader_test(tw, qw, i, j, transition) == want, (i, j)
        n_match += want
    assert n_match > 100


@pytest.mark.parametrize('X', [251, 910, 6399])
def test_windows_give_the_reference_best_termination_and_cells(X):
    """Both sides of a hit through the kernel's windows (the batch's block for right window 0 and left window 0, the later
    windows read on their own), against scan_reference.xdrop_side: best, whether the side is still open, and the chunks
    counted, with non-ACGT columns inside the windows."""
    T, Q = related_pair(X)
    tw, qw = plane_words(T), plane_words(Q)
    tab = [s1_entry(i, X) for i in range(4096)]
    rng = np.random.default_rng(X + 1)
    I = rng.integers(R.END_PAD + 100, R.END_PAD + 5850, 400)
    J = I + rng.integers(-2, 3, 400)
    ref_r = R.xdrop_side(R.side_columns(T, Q, I, J, True), X)
    ref_l = R.xdrop_side(R.side_columns(T, Q, I, J, False), X)
    n_slow = 0
    for h, (i, j) in enumerate(zip(I.tolist(), J.tolist())):
        m = [nib_merge(a, b) for a, b in zip(nib_span(tw, i - 13, 8), nib_span(qw, j - 13, 8))]
        windows = {True: [m[4:8]], False: [[nib_rev(m[3 - k]) for k in range(4)]]}
        for right, b in ((True, 1), (False, 1), (False, 2)):
            d = R.SEED_SPAN + 30 * b if right else R.SEED_SPAN - 30 * b - 32
            t, q = nib_span(tw, i + d, 4), nib_span(qw, j + d, 4)
            w = [nib_merge(t[k], q[k]) for k in range(4)]
            windows[right].append(w if right else [nib_rev(w[3 - k]) for k in range(4)])
        for right, ref in ((True, ref_r), (False, ref_l)):
            best, D, chunks = 0, 125, 0
            for w in windows[right]:
                pw, an = s1_prepare(list(w))
                n_slow += an and D < DONE // 2
                best, D, c = xdrop_window30(tab, pw, an, best, D)
                chunks += c
            ncols = 60 if right else 90
            assert best == ref[0][h], (h, right)
            assert (D < DONE // 2) == (ref[1][h] >= ncols), (h, right)
            assert chunks == ref[2][h], (h, right)
    assert n_slow > 20
