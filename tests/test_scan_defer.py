"""The deferred continuation windows of the seed scan (mimeo_b200/csrc/seed.cu), restated with Python integers. No GPU needed.

A batch of 32 hits runs right window 0 and left windows 0 and 1; a hit still open on either side is stored as a 16-byte
record {hi, hj, s1_pack(best_r, D_r), s1_pack(best_l, D_l)} in its warp's queue, and drain batches of up to 32 records run
right window 1 and left window 2. Held against the inline schedule (every window of a batch run by the batch itself):
  * s1_pack / s1_unpack lose nothing over every (best, D) a side can hold for every x-drop the scan accepts;
  * deferring gives the same survivors and, hit for hit, the same number of chunks entered while open (the stage-1 cell
    count), whatever hits share a warp, including the polls that end a window early."""
import numpy as np
import pytest

HOXD70 = np.array([[91, -114, -31, -123], [-114, 100, -125, -31], [-31, -125, 100, -114], [-123, -31, -114, 91]], dtype=np.int64)
SCORE_N = -100
DONE = 1 << 24
D0 = 125
MAX_XDROP = 8191 - 125 - 300
VOTES = 0x148                     # the later windows poll before chunks 3, 6 and 8
M32 = 0xFFFFFFFF


def s1_pack(best, D):
    return best | ((D if D < DONE // 2 else 0xFFFF) << 16)


def s1_unpack(w):
    return w & 0xFFFF, (DONE if (w >> 16) == 0xFFFF else w >> 16)


def window30(lanes, side, w, X, votes):
    """xdrop_window30 for a warp: lanes = list of hit states, side 'r' / 'l', w = window index. Updates best, D, chunks."""
    for s in lanes:
        s['_n'] = 0
        cols = s[side + 'cols'][30 * w:30 * w + 30]
        best, D = s['best_' + side], s['D_' + side]
        if D < DONE // 2 and (cols == SCORE_N).any():              # the per-column path of a window with a non-ACGT column
            run, term = best - (D - 125), False
            for sc in cols.tolist():
                run += sc
                if run > best:
                    best = run
                elif run < best - X:
                    term = True
                    break
            s['_n'] = 10
            s['_keep'] = DONE if term else (best - run) + 125
            s['best_' + side], s['D_' + side] = best, DONE
        else:
            s['_keep'] = None
    entered, parked = 10, [0] * len(lanes)
    for k in range(10):
        if (votes >> k) & 1 and all(s['D_' + side] >= DONE // 2 for s in lanes):
            entered = k
            break
        for i, s in enumerate(lanes):
            c = s[side + 'cols'][30 * w + 3 * k:30 * w + 3 * k + 3]
            p = np.cumsum(c)
            sm, mx, mn = int(p[-1]), int(p.max()), int(p.min())
            D = s['D_' + side]
            parked[i] += D
            term = mn + X + 125 < D
            dm = max(D, mx + 125)
            s['best_' + side] += dm - D
            s['D_' + side] = DONE if term else dm - sm
    for i, s in enumerate(lanes):
        s['chunks'] += s['_n'] + entered - (parked[i] >> 24)
        if s['_keep'] is not None:
            s['D_' + side] = s['_keep']


def fresh(hit, live):
    return dict(hit, best_r=0, best_l=0, D_r=D0 if live else DONE, D_l=D0 if live else DONE, chunks=0)


def is_open(D):
    return D < DONE // 2


def survivor(s, K):
    return is_open(s['D_r']) or is_open(s['D_l']) or s['best_r'] + s['best_l'] >= K


def inline_schedule(hits, X, K):
    out = {}
    for b in range(0, len(hits), 32):
        lanes = [fresh(h, True) for h in hits[b:b + 32]]
        window30(lanes, 'r', 0, X, 0)
        if not all(not is_open(s['D_r']) for s in lanes):
            window30(lanes, 'r', 1, X, VOTES)
        window30(lanes, 'l', 0, X, 0)
        for w in (1, 2):
            if all(not is_open(s['D_l']) for s in lanes):
                break
            window30(lanes, 'l', w, X, VOTES)
        for s in lanes:
            out[s['id']] = (survivor(s, K), s['chunks'])
    return out


def deferred_schedule(hits, X, K, order):
    """order: the sequence in which hits reach the scan (which hits share a batch); drains as the kernel schedules them.
    Returns the per-hit results and the number of hits that went through the queue."""
    out, queue, head = {}, {}, 0
    tail = 0
    byid = {h['id']: h for h in hits}
    seq = [byid[i] for i in order]
    pos = 0
    while True:
        pending, queued = len(seq) - pos, tail - head
        if pending == 0 and queued == 0:
            break
        if queued >= 32 or pending == 0:
            nd = min(queued, 32)
            lanes = []
            for r in range(nd):
                rec = queue.pop((head + r) % 64)
                s = fresh(byid[rec[0]], True)
                assert rec[1] == s['hj']
                s['best_r'], s['D_r'] = s1_unpack(rec[2])
                s['best_l'], s['D_l'] = s1_unpack(rec[3])
                s['chunks'] = rec[4]
                lanes.append(s)
            head += nd
            lanes += [fresh(byid[seq[0]['id']], False) for _ in range(32 - nd)]   # idle lanes: parked, never counted
            if not all(not is_open(s['D_r']) for s in lanes):
                window30(lanes, 'r', 1, X, VOTES)
            if not all(not is_open(s['D_l']) for s in lanes):
                window30(lanes, 'l', 2, X, VOTES)
            for s in lanes[:nd]:
                out[s['id']] = (survivor(s, K), s['chunks'])
            for s in lanes[nd:]:
                assert s['chunks'] == 0
        else:
            lanes = [fresh(h, True) for h in seq[pos:pos + 32]]
            pos += len(lanes)
            window30(lanes, 'r', 0, X, 0)
            window30(lanes, 'l', 0, X, 0)
            if not all(not is_open(s['D_l']) for s in lanes):
                window30(lanes, 'l', 1, X, VOTES)
            for s in lanes:
                if is_open(s['D_r']) or is_open(s['D_l']):
                    assert (tail + 1) - head <= 64                          # the queue never overruns its 64 slots
                    queue[tail % 64] = (s['id'], s['hj'], s1_pack(s['best_r'], s['D_r']), s1_pack(s['best_l'], s['D_l']), s['chunks'])
                    tail += 1
                else:
                    out[s['id']] = (s['best_r'] + s['best_l'] >= K, s['chunks'])
    return out, tail


def make_hits(rng, n):
    """seed hits: the left side starts with the 19 seed columns (12 care positions match), the rest random or related
    (substitutions at a random rate, so that some extensions stay open through all windows), now and then a non-ACGT column"""
    hits = []
    for i in range(n):
        t = rng.integers(0, 4, 150)
        kind = rng.random()
        rate = 0.75 if kind < 0.7 else rng.uniform(0.02, 0.4)
        q = np.where(rng.random(150) < rate, rng.integers(0, 4, 150), t)
        q[60:79] = np.where(rng.random(19) < 0.3, q[60:79], t[60:79])
        sc = HOXD70[t, q]
        if rng.random() < 0.05:
            sc[rng.integers(0, 150, int(rng.integers(1, 4)))] = SCORE_N
        right = sc[79:139].copy()                      # hit + 19 onwards
        left = sc[:79][::-1].copy()                    # last seed column downwards: 19 seed + 60 flank
        left = np.concatenate([left, HOXD70[rng.integers(0, 4, 11), rng.integers(0, 4, 11)]])
        hits.append({'id': i, 'hj': int(rng.integers(0, 1 << 32)), 'rcols': right, 'lcols': left})
    return hits


def test_record_pack_is_lossless():
    for best in list(range(0, 200)) + list(range(9000 - 200, 9001)) + [(1 << 16) - 1]:
        for D in [125, 126, 1035, 7766 + 125, (1 << 13) - 1, DONE]:
            w = s1_pack(best, D)
            assert 0 <= w <= M32
            assert s1_unpack(w) == (best, D)
    rng = np.random.default_rng(3)
    for _ in range(20000):
        X = int(rng.integers(251, MAX_XDROP + 1))
        best = int(rng.integers(0, 90 * 100 + 1))
        D = DONE if rng.random() < 0.2 else int(rng.integers(125, X + 126))
        assert s1_unpack(s1_pack(best, D)) == (best, D)


@pytest.mark.parametrize('X,K', [(910, 3000), (251, 2000), (1500, 3500)])
def test_deferred_windows_equal_inline(X, K):
    rng = np.random.default_rng(X)
    hits = make_hits(rng, 32 * 40 + 7)
    want = inline_schedule(hits, X, K)
    n_surv = sum(s for s, _ in want.values())
    assert 0 < n_surv < len(hits)
    for trial in range(2):
        order = [h['id'] for h in hits] if trial == 0 else rng.permutation(len(hits)).tolist()
        got, n_deferred = deferred_schedule(hits, X, K, order)
        assert n_deferred > 64                          # several full drains were exercised
        assert got == want                              # per hit: survivor decision and chunks entered while open
