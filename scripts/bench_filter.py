"""Measures `mimeo filter` on a seeded library shaped like repeat segments extracted from `mimeo x` / `self` output: 50 000
records of log-uniform length over 100 bp - 20 kbp plus six of 100 - 500 kbp; about a third carry one planted microsatellite
(period 1-50, 10-90 % of the record, 0-5 % substitutions, some soft-masked, some broken by N runs).

One command, one JSON document (stdout and --out), at default mask parameters and --maxtandem 40: card name, power limit and
max SM clock; records, bases and strip cells (2 * sum over records of the cells of one pass); end-to-end wall time of
`run_filter.main` (FASTA on disk -> files written) with and without --writeTRF; the `tandem_mask` kernel time from mb2_prof
(separate runs) with and without runs, GCUPS; the longest record alone and its share; records dropped; the C oracle on a
sample of records plus the longest one, and whether every masked count and run of the sample agrees. The `--reportTRF` leg:
end-to-end wall time with --reportTRF, the `tandem_report` kernel time next to `tandem_mask` in the same call and its share,
and whether the counts equal the mask's and every run's report of the sample equals the report oracle.

    python scripts/bench_filter.py --steps 3 --warmup 1 --out profiles/r5_filter_library.json
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'scripts'))

from bench_tandem import strip_cells  # noqa: E402


def repeat_library(seed=2025, n=50_000, nbig=6, sat_frac=1 / 3):
    rng = np.random.default_rng(seed)
    bases = np.frombuffer(b'ACGT', dtype=np.uint8)
    lens = np.exp(rng.uniform(np.log(100), np.log(20_000), n)).astype(np.int64)
    lens = np.insert(lens, rng.integers(0, n, nbig), rng.integers(100_000, 500_001, nbig))
    recs = []
    for k, L in enumerate(lens.tolist()):
        s = bases[rng.integers(0, 4, L)]
        if rng.random() < sat_frac:
            d = int(rng.integers(1, 51))
            alen = max(d, int(rng.uniform(0.1, 0.9) * L))
            arr = np.resize(bases[rng.integers(0, 4, d)], alen)
            sub = rng.random(alen) < float(rng.choice([0.0, 0.02, 0.05]))
            arr[sub] = bases[rng.integers(0, 4, int(sub.sum()))]
            if rng.random() < 0.3:
                arr = arr + np.uint8(32)                                       # soft-masked
            if rng.random() < 0.3:
                for _ in range(int(rng.integers(1, 4))):                       # broken by N runs
                    at, nl = int(rng.integers(0, alen)), int(rng.integers(1, 30))
                    arr[at:at + nl] = ord('N')
            at = int(rng.integers(0, L - alen + 1))
            s[at:at + alen] = arr
        recs.append((f'seg{k:06d} len={L}', s))
    return recs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=1)
    ap.add_argument('--sample', type=int, default=300, help='records checked against the C oracle (plus the longest one)')
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    from mimeo_b200 import _lib, run_filter, tandem
    from mimeo_b200.fasta import write_fasta_record
    from oracle import tandem_oracle as to
    from tests import tandem_report_reference as trr
    smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True, text=True)
    card = smi.stdout.strip().splitlines()[0] if smi.returncode == 0 and smi.stdout.strip() else torch.cuda.get_device_name(0)
    t0 = time.perf_counter()
    recs = repeat_library()
    t_gen = time.perf_counter() - t0
    seqs = [s for _h, s in recs]
    lens = np.array([len(s) for s in seqs], dtype=np.int64)
    p = tandem.params()
    maxtandem = 40.0
    res = {'what': 'mimeo filter on a seeded repeat-segment library (50 000 records log-uniform 100 bp - 20 kbp + 6 of 100-500 kbp, '
                   'a third with a planted microsatellite of period 1-50 over 10-90 % of the record), default mask parameters, '
                   '--maxtandem 40',
           'card': card, 'steps': args.steps, 'warmup': args.warmup, 'generate_s': t_gen,
           'records': len(recs), 'bases': int(lens.sum()), 'longest_record_bp': int(lens.max()),
           'cells_both_passes': 2 * strip_cells(lens, p['maxperiod'])}
    with tempfile.TemporaryDirectory() as tmp:
        infile = os.path.join(tmp, 'library.fa')
        with open(infile, 'wb') as f:
            for h, s in recs:
                write_fasta_record(f, h, s, width=80)
        res['input_fasta_bytes'] = os.path.getsize(infile)
        _lib.init()
        for key, extra in (('e2e_ms', []), ('e2e_writetrf_ms', ['--writeTRF']), ('e2e_reporttrf_ms', ['--reportTRF'])):
            wall = []
            for k in range(args.warmup + args.steps):
                sys.argv = ['mimeo-filter', '--infile', infile, '-d', os.path.join(tmp, 'out'), '--loglevel', 'WARNING'] + extra
                _lib.sync()
                t0 = time.perf_counter()
                run_filter.main()
                _lib.sync()
                if k >= args.warmup:
                    wall.append(1e3 * (time.perf_counter() - t0))
            res[key] = wall
        with open(os.path.join(tmp, 'out', 'mimeo_filtered.fa'), 'rb') as f:
            res['records_kept_in_outfile'] = f.read().count(b'>')

    _lib.prof_enable(True)

    def kernel_ms(xs, runs):
        out, ms = None, []
        for k in range(args.warmup + args.steps):
            _lib.prof_reset()
            out = tandem.record_masks(xs, p, runs=runs)
            _lib.sync()
            t, batches = _lib.prof_get('tandem_mask')
            if k >= args.warmup:
                ms.append(t)
        return out, ms, batches

    (m, _), res['tandem_mask_kernel_ms'], res['launches'] = kernel_ms(seqs, False)
    (m_runs, runs), res['tandem_mask_runs_kernel_ms'], _ = kernel_ms(seqs, True)
    li = int(np.argmax(lens))
    _, res['longest_record_kernel_ms'], _ = kernel_ms([seqs[li]], False)
    res['report_call_tandem_mask_kernel_ms'], res['tandem_report_kernel_ms'] = [], []
    for k in range(args.warmup + args.steps):
        _lib.prof_reset()
        m_rep, reps = tandem.record_reports(seqs, p)
        _lib.sync()
        if k >= args.warmup:
            res['report_call_tandem_mask_kernel_ms'].append(_lib.prof_get('tandem_mask')[0])
            res['tandem_report_kernel_ms'].append(_lib.prof_get('tandem_report')[0])
    _lib.prof_enable(False)
    kmed = float(np.median(res['tandem_mask_kernel_ms']))
    res['gcups_kernel_median'] = res['cells_both_passes'] / (kmed * 1e-3) / 1e9
    res['longest_record_share_of_kernel'] = float(np.median(res['longest_record_kernel_ms'])) / kmed
    drop = 100.0 * m.astype(np.float64) / np.maximum(lens, 1) > maxtandem
    res['records_dropped'] = int(drop.sum())
    res['masked_bp'] = int(m.sum())
    res['counts_equal_with_and_without_runs'] = bool((m == m_runs).all())
    res['report_runs'] = int(sum(len(rr) for rr in reps))
    res['report_kernel_over_mask_kernel'] = float(np.median(res['tandem_report_kernel_ms'])) / float(np.median(res['report_call_tandem_mask_kernel_ms']))
    res['e2e_reporttrf_over_e2e'] = float(np.median(res['e2e_reporttrf_ms'])) / float(np.median(res['e2e_ms']))
    # the C oracle on a sample of records plus the longest one, single-threaded
    rng = np.random.default_rng(7)
    sample = sorted(set(rng.choice(len(recs), args.sample, replace=False).tolist()) | {li})
    t0 = time.perf_counter()
    want = {k: to.mask(seqs[k], **p) for k in sample}
    res['oracle_sample_records'] = len(sample)
    res['oracle_sample_bp'] = int(lens[sample].sum())
    res['oracle_s_single_thread'] = time.perf_counter() - t0
    res['oracle_sample_cells'] = 2 * strip_cells(lens[sample], p['maxperiod'])
    res['gpu_matches_oracle_on_sample'] = all((int(m[k]), runs[k]) == want[k] for k in sample)
    res['report_gpu_matches_oracle_on_sample'] = bool((m_rep == m).all()) and all(
        [(r.start, r.end) for r in reps[k]] == runs[k] and all(trr.report(seqs[k][r.start:r.end + 1], **p) == tuple(r[2:]) for r in reps[k])
        for k in sample)
    res['records_kept_in_outfile_matches'] = res['records_kept_in_outfile'] == len(recs) - res['records_dropped']
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(txt + '\n')
    assert res['gpu_matches_oracle_on_sample'] and res['counts_equal_with_and_without_runs'], 'GPU mask differs from the oracle'
    assert res['report_gpu_matches_oracle_on_sample'], 'GPU tandem report differs from the oracle'


if __name__ == '__main__':
    main()
