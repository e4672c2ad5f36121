"""Exact CPU statement of the seed scan's first stage (mimeo_b200/csrc/seed.cu, seed_scan_kernel), the reference the survivor
list of `mb2_test_seed_scan` is held to. numpy and Python integers only; no GPU needed.

Everything happens in the padded coordinate space of a device genome (seq.cuh): scaffold s occupies [off[s], off[s] + len[s]),
every other position is pad. Pads and non-ACGT bases score SCORE_N in every column; soft-masked (lower-case) bases score by
their base but are never part of a seed word.

  * seed hits   every seedable 19-mer window of the query (positions [END_PAD, G_Q - END_PAD)) is looked up 13 times
                (once when transition = 0): its 24-bit key of the 12 care bases, and the key with the transition bit of one
                care base flipped. Every seedable target window with that key is a hit (i, j).
  * leaders     a hit is a run leader iff (i - 1, j - 1) is not a seed hit (spec D1).
  * extension   per leader, the column x-drop rule (run += score; a new maximum raises best, else run < best - X ends it)
                over 60 columns to the right (from i + 19) and 90 to the left (from i + 18 downwards, through the seed).
  * survivors   a leader survives iff the right side is still open after its 60 columns, or the left side after its 90, or
                best_r + best_l >= K.
  * cells       stage1_cells = 3 x the three-column chunks a leader entered while still open. A side is cut into windows of
                30 columns (10 chunks); a window with a non-ACGT column that is entered while open takes the per-column path
                and counts all 10 chunks.
"""
from __future__ import annotations

from typing import Dict, Sequence

import numpy as np

from oracle import lastz_oracle as lo

GENOME_PAD = 64
END_PAD = 2048
SEED_SPAN = 19
SCORE_N = -100
CARE = (0, 1, 2, 4, 7, 8, 11, 13, 15, 16, 17, 18)
WINDOW = 30
RIGHT_COLS = 60
LEFT_COLS = 90
HOXD70 = np.array([[91, -114, -31, -123], [-114, 100, -125, -31], [-31, -125, 100, -114], [-123, -31, -114, 91]], dtype=np.int32)
KEY_BITS = 2 * len(CARE)
HIGH_BITS = int('10' * len(CARE), 2)          # the transition bit of every care base in a key


def layout(lengths: Sequence[int]):
    """Scaffold offsets and padded length G of a genome of these scaffold lengths (genome.cu: layout)."""
    off, pos = [], END_PAD
    for n in lengths:
        off.append(pos)
        pos = (pos + int(n) + GENOME_PAD + 63) & ~63
    return np.array(off, dtype=np.int64), pos + END_PAD


class Space:
    """One genome in padded coordinates: base (0..3, 0 where bad), bad (non-ACGT or pad), noseed (bad or soft-masked),
    key (seed key of the window starting there) and seedable (the window holds no noseed position). Arrays hold G + 64
    positions, as the device arrays do."""

    def __init__(self, codes: Sequence[np.ndarray], off=None):
        codes = [np.asarray(c, dtype=np.uint8) for c in codes]
        lengths = [len(c) for c in codes]
        want_off, G = layout(lengths)
        if off is not None:
            assert list(np.asarray(off)) == list(want_off), 'scaffold offsets differ from the layout rule'
        self.off, self.len, self.G = want_off, np.array(lengths, dtype=np.int64), G
        n = G + 64
        self.base = np.zeros(n, dtype=np.int64)
        self.bad = np.ones(n, dtype=bool)
        self.noseed = np.ones(n, dtype=bool)
        for o, c in zip(want_off, codes):
            b = c & 7
            self.bad[o:o + len(c)] = b > 3
            self.base[o:o + len(c)] = np.where(b > 3, 0, b)
            self.noseed[o:o + len(c)] = (b > 3) | ((c & 8) != 0)
        ns = np.concatenate([[0], np.cumsum(self.noseed)])
        p = np.arange(n - SEED_SPAN + 1)
        self.seedable = np.zeros(n, dtype=bool)
        self.seedable[p] = ns[p + SEED_SPAN] == ns[p]
        self.key = np.zeros(n, dtype=np.int64)
        for k, c in enumerate(CARE):
            self.key[p] |= self.base[p + c] << (2 * k)

    @classmethod
    def from_ascii(cls, seqs: Sequence, off=None, revcomp=False) -> 'Space':
        codes = [lo.encode(s) for s in seqs]
        if revcomp:
            codes = [lo.revcomp_codes(c) for c in codes]
        return cls(codes, off)

    def scaffold_of(self, p):
        """Scaffold index of padded positions p (-1 inside a pad)."""
        p = np.asarray(p)
        s = np.searchsorted(self.off, p, side='right') - 1
        ok = (s >= 0) & (p < self.off[np.maximum(s, 0)] + self.len[np.maximum(s, 0)])
        return np.where(ok, s, -1)


def keys_match(a, b, transition):
    """seed_match on two keys: equal on every care base, or (transition) different in one transition bit only."""
    x = a ^ b
    one_bit = (x != 0) & ((x & (x - 1)) == 0) & ((x & ~HIGH_BITS) == 0)
    return (x == 0) | (one_bit if transition else False)


def seed_hits(T: Space, Q: Space, transition: int):
    """All seed hits (i, j) as two int64 arrays, in no particular order."""
    tpos = np.flatnonzero(T.seedable[:T.G])
    order = np.argsort(T.key[tpos], kind='stable')
    tpos = tpos[order]
    tkeys = T.key[tpos]
    qpos = np.arange(END_PAD, Q.G - END_PAD)
    qpos = qpos[Q.seedable[qpos]]
    qkey = Q.key[qpos]
    flips = [0] + ([2 << (2 * k) for k in range(len(CARE))] if transition else [])
    I, J = [], []
    for f in flips:
        kk = qkey ^ f
        a = np.searchsorted(tkeys, kk, side='left')
        b = np.searchsorted(tkeys, kk, side='right')
        cnt = b - a
        tot = int(cnt.sum())
        if tot == 0:
            continue
        starts = np.repeat(a - (np.cumsum(cnt) - cnt), cnt)
        I.append(tpos[starts + np.arange(tot)])
        J.append(np.repeat(qpos, cnt))
    if not I:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    return np.concatenate(I), np.concatenate(J)


def is_leader(T: Space, Q: Space, I, J, transition):
    pred = T.seedable[I - 1] & Q.seedable[J - 1] & keys_match(T.key[I - 1], Q.key[J - 1], transition)
    return ~pred


def side_columns(T: Space, Q: Space, I, J, right: bool):
    """Column scores of one side of every hit in extension order: (n, 60) right, (n, 90) left."""
    if right:
        c = np.arange(RIGHT_COLS)
        ti, qj = I[:, None] + SEED_SPAN + c, J[:, None] + SEED_SPAN + c
    else:
        c = np.arange(LEFT_COLS)
        ti, qj = I[:, None] + SEED_SPAN - 1 - c, J[:, None] + SEED_SPAN - 1 - c
    bad = T.bad[ti] | Q.bad[qj]
    return np.where(bad, SCORE_N, HOXD70[T.base[ti], Q.base[qj]]).astype(np.int32)


def xdrop_side(sc, X):
    """Vectorised column x-drop over the bounded columns of one side: (best, termination column or ncols, chunks entered
    while open)."""
    n, ncols = sc.shape
    run = np.cumsum(sc, axis=1, dtype=np.int64)
    best_incl = np.maximum(np.maximum.accumulate(run, axis=1), 0)
    term = run < best_incl - X
    has = term.any(axis=1)
    tcol = np.where(has, np.argmax(term, axis=1), ncols)
    best = best_incl[np.arange(n), np.minimum(tcol, ncols - 1)]
    chunks = np.zeros(n, dtype=np.int64)
    for w in range(ncols // WINDOW):
        entered = tcol >= WINDOW * w
        slow = (sc[:, WINDOW * w:WINDOW * (w + 1)] == SCORE_N).any(axis=1)
        inside = np.minimum((tcol - WINDOW * w) // 3 + 1, WINDOW // 3)
        chunks += np.where(entered, np.where(slow, WINDOW // 3, inside), 0)
    return best, tcol, chunks


def leaders(T: Space, Q: Space, transition: int):
    """(number of seed hits, target and query positions of the run leaders)."""
    I, J = seed_hits(T, Q, transition)
    lead = is_leader(T, Q, I, J, transition)
    return len(I), I[lead], J[lead]


def first_stage(T: Space, Q: Space, X: int, transition: int, lead=None, batch: int = 1 << 18) -> Dict[str, np.ndarray]:
    """The scan's first stage for every leader (lead = a result of leaders() to reuse). Returns the hit count and, per
    leader: i, j, best_r, best_l, tcol_r, tcol_l (termination column, or 60 / 90 when still open) and chunks."""
    nhits, I, J = lead if lead is not None else leaders(T, Q, transition)
    out = {'seed_hits': nhits, 'i': I, 'j': J}
    parts = {k: [] for k in ('best_r', 'tcol_r', 'best_l', 'tcol_l', 'chunks')}
    for a in range(0, len(I), batch):
        i, j = I[a:a + batch], J[a:a + batch]
        br, tr, cr = xdrop_side(side_columns(T, Q, i, j, True), X)
        bl, tl, cl = xdrop_side(side_columns(T, Q, i, j, False), X)
        for k, v in (('best_r', br), ('tcol_r', tr), ('best_l', bl), ('tcol_l', tl), ('chunks', cr + cl)):
            parts[k].append(v)
    for k, v in parts.items():
        out[k] = np.concatenate(v) if v else np.zeros(0, np.int64)
    return out


def survivors(fs: Dict[str, np.ndarray], K: int):
    """Boolean mask of the surviving leaders of first_stage() at score threshold K."""
    return (fs['tcol_r'] >= RIGHT_COLS) | (fs['tcol_l'] >= LEFT_COLS) | (fs['best_r'] + fs['best_l'] >= K)


def summary(fs: Dict[str, np.ndarray], K: int):
    """(sorted survivor list as (n, 2) [i, j], counters [survivors, seed hits, leaders, stage-1 cells])."""
    m = survivors(fs, K)
    surv = np.stack([fs['i'][m], fs['j'][m]], axis=1)
    surv = surv[np.lexsort((surv[:, 1], surv[:, 0]))] if len(surv) else surv.reshape(0, 2)
    return surv, [int(m.sum()), int(fs['seed_hits']), int(len(fs['i'])), 3 * int(fs['chunks'].sum())]


def deferred(fs: Dict[str, np.ndarray]):
    """Leaders a batch of the kernel hands to the deferred queue: still open on the right after right window 0 or on the left
    after left window 1."""
    return (fs['tcol_r'] >= WINDOW) | (fs['tcol_l'] >= 2 * WINDOW)


# ------------------------------------------------------------------------------------------ plain per-hit statement
def brute_hit(T: Space, Q: Space, i: int, j: int, X: int, transition: int):
    """One hit, column by column with Python integers and no numpy vector logic: (is leader, best_r, open_r, best_l, open_l,
    chunks). Used to check the vectorised statement above."""
    def seedable(S, p):
        return all(not S.noseed[p + c] for c in range(SEED_SPAN))

    def key(S, p):
        return sum(int(S.base[p + c]) << (2 * k) for k, c in enumerate(CARE))

    pred = seedable(T, i - 1) and seedable(Q, j - 1)
    if pred:
        diffs = [(int(T.base[i - 1 + c]), int(Q.base[j - 1 + c])) for c in CARE]
        nd = [(a, b) for a, b in diffs if a != b]
        pred = not nd or (bool(transition) and len(nd) == 1 and (nd[0][0] ^ nd[0][1]) == 2)
    if pred:
        return (False, 0, False, 0, False, 0)
    res, chunks = [], 0
    for ncols, step, ti, qj in ((RIGHT_COLS, 1, i + SEED_SPAN, j + SEED_SPAN), (LEFT_COLS, -1, i + SEED_SPAN - 1, j + SEED_SPAN - 1)):
        run = best = 0
        is_open = True
        for w in range(ncols // WINDOW):
            if not is_open:
                break
            cols = [(ti + step * c, qj + step * c) for c in range(WINDOW * w, WINDOW * (w + 1))]
            slow = any(T.bad[a] or Q.bad[b] for a, b in cols)
            if slow:
                chunks += WINDOW // 3
            for c, (a, b) in enumerate(cols):
                if not slow and c % 3 == 0:
                    chunks += 1                    # the table path enters this chunk while open
                sc = SCORE_N if (T.bad[a] or Q.bad[b]) else int(HOXD70[T.base[a], Q.base[b]])
                run += sc
                if run > best:
                    best = run
                elif run < best - X:
                    is_open = False
                    break
        res += [best, is_open]
    return (True, res[0], res[1], res[2], res[3], chunks)


# ------------------------------------------------------------------------------------------ test genomes
def _acgt(rng, n):
    return np.frombuffer(b'ACGT', dtype=np.uint8)[rng.integers(0, 4, n)].copy()


def scan_genome(kind: str) -> Dict[str, np.ndarray]:
    """Small genomes ({name: uint8 ASCII}) that reach the scan's awkward paths:
      repeats  ordinary planted repeats with N runs
      soft     the same with lower-case (soft-masked) stretches
      edges    scaffold lengths with len % 64 in {0, 51, 63} (pads of exactly 64 columns) and tiny scaffolds of 1-65 bases
               cut from scaffold ends, so that hits sit right at scaffold edges; the last scaffold's length is not a
               multiple of 32, so the query's last round of 32 positions is partial
      dense    a 10 kbp tandem array of period 6-12 and an (AC)n run: thousands of hits per query position
      family   one family of 1 kbp copies at 70-85 % pairwise identity: many hits still open after the first windows"""
    from tests.helpers import mutate, synth_genome
    rng = np.random.default_rng(sum(map(ord, kind)))
    if kind == 'repeats':
        return synth_genome(501, 3, 20_000, 3, copies=(3, 6), fam_len=(300, 1500), sub=0.08, indel=0.004, n_runs=6)
    if kind == 'soft':
        g = synth_genome(502, 2, 25_000, 3, copies=(4, 7), fam_len=(400, 1500), sub=0.08, indel=0.004, n_runs=2)
        for s in g.values():
            for _ in range(8):
                p0 = int(rng.integers(0, len(s) - 1600))
                s[p0:p0 + int(rng.integers(20, 1500))] |= 0x20
        return g
    if kind == 'edges':
        a, b, c = _acgt(rng, 6400), _acgt(rng, 6451), _acgt(rng, 6463)
        b[:300] = a[-300:]                                   # the end of one scaffold repeats at the start of the next
        c[-300:] = mutate(rng, a[:300], 0.05, 0.0)               # and, diverged, at the end of a third
        g = {'a': a, 'b': b, 'c': c}
        for n in (1, 18, 19, 20, 63, 64, 65):
            g[f'head{n}'] = a[:n].copy()
            g[f'tail{n}'] = b[len(b) - n:].copy()
        g['last'] = np.concatenate([a[100:2100], _acgt(rng, 1013)])   # 3013 bases: 3013 % 32 = 5
        return g
    if kind == 'dense':
        unit = _acgt(rng, int(rng.integers(6, 13)))
        arr = np.tile(unit, 10_000 // len(unit) + 1)[:10_000].copy()
        ac = np.tile(np.frombuffer(b'AC', dtype=np.uint8), 1000)
        return {'tandem': np.concatenate([_acgt(rng, 2000), arr, _acgt(rng, 2000), ac, _acgt(rng, 1000)]),
                'other': np.concatenate([_acgt(rng, 3000), mutate(rng, arr[:600], 0.03, 0.0), _acgt(rng, 3000)])}
    if kind == 'family':
        cons = _acgt(rng, 1000)
        parts = []
        for _ in range(40):
            parts += [_acgt(rng, int(rng.integers(50, 400))), mutate(rng, cons, float(rng.uniform(0.08, 0.15)), 0.002)]
        return {'fam': np.concatenate(parts + [_acgt(rng, 500)])}
    raise ValueError(kind)


SCAN_GENOMES = ('repeats', 'soft', 'edges', 'dense', 'family')
