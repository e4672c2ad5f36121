"""Measures the tandem-repeat mask of `mimeo map --maxtandem` on the C3 map job (tests/helpers.py:synth_c3's generator)
with microsatellites planted in A before B is derived from it, so that the filter drops a real share of hits.

One command, one JSON document (stdout and --out): card name and power limit; the map step (alignment + device filter)
and the mask per step with CUDA events (`tandem_mask` tag) after a warm-up; cells (2 * sum of strip cells over distinct
spans), GCUPS, spans, distinct spans, rows dropped at --maxtandem; the longest span alone; the C oracle on the same spans
and whether every masked count agrees. The `--reportTRF` leg: the call that computes the mask and the report together
(`tandem_report` tag next to `tandem_mask`), the report kernel's share of the mask kernel, and whether its counts equal the
mask's and every run's report equals the report oracle (tests/tandem_report_oracle.c).

    python scripts/bench_tandem.py --steps 5 --warmup 1 --out profiles/r4_tandem_c3.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def c3_with_microsatellites(seed=1003, nscaf=40, scaf_len=1_000_000, block=50_000, keep_frac=0.60, sub=0.08, indel=0.005, inv_frac=0.10,
                            sat_seed=4004, sats_per_mbp=60):
    """synth_c3 with exact microsatellites (period 1..12, 40..400 bp) planted in A before B is derived from it."""
    from tests.helpers import mutate, revcomp_ascii
    rng = np.random.default_rng(seed)
    srng = np.random.default_rng(sat_seed)
    bases = np.frombuffer(b'ACGT', dtype=np.uint8)
    A, B = {}, {}
    for i in range(nscaf):
        a = bases[rng.integers(0, 4, scaf_len)]
        for _ in range(int(sats_per_mbp * scaf_len / 1e6)):
            unit = bases[srng.integers(0, 4, int(srng.integers(1, 13)))]
            n = int(srng.integers(40, 401))
            at = int(srng.integers(0, scaf_len - n))
            a[at:at + n] = np.resize(unit, n)
        parts = []
        for p in range(0, scaf_len, block):
            blk = a[p:p + block]
            if rng.random() < keep_frac:
                m = mutate(rng, blk, sub, indel)
                parts.append(revcomp_ascii(m) if rng.random() < inv_frac else m)
            else:
                parts.append(bases[rng.integers(0, 4, len(blk))])
        A[f'A{i:03d}'] = a
        B[f'B{i:03d}'] = np.concatenate(parts)
    return A, B


def strip_cells(n, P):
    """Cells of one pass over a span of length n: pairs (i, j), 1 <= i < j <= n, j - i <= P."""
    n = np.asarray(n, dtype=np.int64)
    d = np.minimum(P, np.maximum(n - 1, 0))
    return int((d * n - d * (d + 1) // 2).sum())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=1)
    ap.add_argument('--maxtandem', type=float, default=40.0)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    from mimeo_b200 import _lib, align as A, tandem
    from mimeo_b200.genome import Genome, align_params
    from oracle import tandem_oracle as to
    from tests import tandem_report_reference as trr
    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True, text=True)
    card = smi.stdout.strip().splitlines()[0] if smi.returncode == 0 and smi.stdout.strip() else torch.cuda.get_device_name(0)
    a, b = c3_with_microsatellites()
    an, bn = sorted(a), sorted(b)
    T, Q = Genome(an, [a[n] for n in an]), Genome(bn, [b[n] for n in bn])
    p = tandem.params()
    _lib.prof_enable(True)

    def map_step():
        dh = A.align_device(T, Q, align_params(3000))
        try:
            dh.filter_sort(100, 90, map_rule=True)
            return dh.download()[0]
        finally:
            dh.close()

    t_map = []
    for k in range(args.warmup + args.steps):
        _lib.sync()
        t0 = time.perf_counter()
        hits = map_step()
        _lib.sync()
        if k >= args.warmup:
            t_map.append(time.perf_counter() - t0)
    scaf = hits['t_id'].astype(np.int32)
    start0 = hits['start1'].astype(np.int64) - 1
    length = hits['end1'].astype(np.int64) - hits['start1'] + 1
    uniq = np.unique(np.stack([scaf, start0, length], 1), axis=0)
    cells = 2 * strip_cells(uniq[:, 2], p['maxperiod'])

    def timed(s, b0, ln, steps, warmup):
        wall, kern = [], []
        m = None
        for k in range(warmup + steps):
            _lib.prof_reset()
            _lib.sync()
            t0 = time.perf_counter()
            m = tandem.masked_counts(T, s, b0, ln, p)
            _lib.sync()
            ms, _ = _lib.prof_get('tandem_mask')
            if k >= warmup:
                wall.append(1e3 * (time.perf_counter() - t0))
                kern.append(ms)
        return m, wall, kern

    m, wall, kern = timed(scaf, start0, length, args.steps, args.warmup)
    rwall, rmask, rkern = [], [], []
    for k in range(args.warmup + args.steps):
        _lib.prof_reset()
        _lib.sync()
        t0 = time.perf_counter()
        rm, reps = tandem.masked_reports(T, scaf, start0, length, p)
        _lib.sync()
        if k >= args.warmup:
            rwall.append(1e3 * (time.perf_counter() - t0))
            rmask.append(_lib.prof_get('tandem_mask')[0])
            rkern.append(_lib.prof_get('tandem_report')[0])
    runs = {(c, s + r.start, r.end - r.start + 1): tuple(r[2:]) for c, s, rr in zip(scaf.tolist(), start0.tolist(), reps) for r in rr}
    t0 = time.perf_counter()
    rep_agree = bool((rm == m).all()) and all(trr.report(a[an[c]][x:x + n], **p) == v for (c, x, n), v in runs.items())
    t_rep_oracle = time.perf_counter() - t0
    drop = 100.0 * m.astype(np.float64) / length > args.maxtandem
    L = int(length.max())
    li = int(np.argmax(length))
    _, lwall, lkern = timed(scaf[li:li + 1], start0[li:li + 1], length[li:li + 1], args.steps, args.warmup)
    # the C oracle on the same distinct spans, single-threaded
    t0 = time.perf_counter()
    om = {}
    for c, s, n in uniq.tolist():
        om[(c, s, n)] = to.mask(a[an[c]][s:s + n], **{k: v for k, v in p.items()})[0]
    t_oracle = time.perf_counter() - t0
    agree = all(int(mm) == om[(c, s, n)] for mm, c, s, n in zip(m.tolist(), scaf.tolist(), start0.tolist(), length.tolist()))
    kmed = float(np.median(kern))
    res = {
        'what': 'tandem-repeat mask of mimeo map --maxtandem on C3 (40 x 1 Mbp A, 60 microsatellites/Mbp of period 1-12 and '
                '40-400 bp planted in A before B is derived), default mask parameters',
        'card': card, 'steps': args.steps, 'warmup': args.warmup,
        'map_step_ms': [1e3 * x for x in t_map],
        'rows': int(len(m)), 'distinct_spans': int(len(uniq)), 'span_bp': int(length.sum()), 'distinct_span_bp': int(uniq[:, 2].sum()),
        'maxtandem': args.maxtandem, 'rows_dropped': int(drop.sum()), 'masked_bp': int(m.sum()),
        'cells_both_passes': cells,
        'tandem_mask_kernel_ms': kern, 'tandem_mask_call_ms': wall,
        'gcups_kernel_median': cells / (kmed * 1e-3) / 1e9 if kmed > 0 else None,
        'filter_over_map_step': float(np.median(wall)) / (1e3 * float(np.median(t_map))),
        'longest_span_bp': L, 'longest_span_kernel_ms': lkern, 'longest_span_call_ms': lwall,
        'oracle_s_single_thread': t_oracle, 'oracle_cells_per_s': cells / t_oracle,
        'gpu_matches_oracle': bool(agree),
        'report_runs': int(sum(len(rr) for rr in reps)), 'report_distinct_runs': len(runs),
        'report_distinct_run_bp': int(sum(n for _c, _x, n in runs)),
        'report_call_ms': rwall, 'report_call_tandem_mask_kernel_ms': rmask, 'tandem_report_kernel_ms': rkern,
        'report_kernel_over_mask_kernel': float(np.median(rkern)) / float(np.median(rmask)),
        'report_call_over_mask_call': float(np.median(rwall)) / float(np.median(wall)),
        'report_oracle_s_single_thread': t_rep_oracle,
        'report_gpu_matches_oracle': rep_agree,
    }
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(txt + '\n')
    T.close(); Q.close()
    assert agree, 'GPU mask differs from the oracle'
    assert rep_agree, 'GPU tandem report differs from the oracle'


if __name__ == '__main__':
    main()
