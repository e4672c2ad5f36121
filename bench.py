#!/usr/bin/env python
"""
bench.py -- measures the hot path on B200 (contract: one JSON line on stdout from rank 0).

  python bench.py --gpus N --steps K --warmup W [--workload x|self|map|cov|c5] [--impl b200|reference] [--dump-outputs DIR]

Default workload = BASELINE config 4 (`mimeo x`, 50 Mbp vs 100 Mbp), the largest named config that fits one GPU within the
driver's time and the one BASELINE.json shards over 8 GPUs; the same job at every N (strong scaling). Configs 1, 2 and 3 are
measured beside it at N=1 (extra keys); config 5 (`--workload c5`, MB2_C5_MBP to scale it down) is run by hand.

A "step" is one pass of the hot path over one batch of synthetic input.
  value : whole-job throughput with inputs already resident in HBM, timed with CUDA events on the
          library's stream, max over ranks.
  e2e   : the same metric through the host-buffer C-ABI call (pinned host memory in, host arrays out,
          H2D/D2H inside the timed region).
  roofline     : the dominant kernel's algorithmic bytes / its CUDA-event time (mb2_prof_*), against
                 MEASURED_PEAKS.json.
  cpu_baseline : the CPU oracle port timed on this box's host cores (rank 0, N=1 only).
--impl reference times the CPU restatement of the reference path (oracle/) with all host threads.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


# ------------------------------------------------------------------------------------------------- helpers
def env_rank():
    return int(os.environ.get('RANK', '0')), int(os.environ.get('LOCAL_RANK', '0')), int(os.environ.get('WORLD_SIZE', '1'))


def measured_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


def ncu_traffic(workload, kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` on this workload, from the committed
    `ncu --set full` capture (profiles/roofline_traffic.json; a number measured under the profiler, so it is only ever
    reported as traffic, never timed). None when no capture of this (workload, kernel) pair is committed."""
    try:
        with open(os.path.join(ROOT, 'profiles', 'roofline_traffic.json')) as f:
            rec = json.load(f)[workload][kernel]
        return rec['dram_bytes_per_launch'], rec['source']
    except Exception:
        return None, None


def ncu_pipes(workload, kernel):
    """Pipe utilisation of `kernel` on this workload from the committed ncu capture (profiles/roofline_traffic.json), or None."""
    try:
        with open(os.path.join(ROOT, 'profiles', 'roofline_traffic.json')) as f:
            return json.load(f)[workload][kernel].get('pipes')
    except Exception:
        return None


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, arrays):
    """Write {name: array} as out_dir/<name>.npy in float64 (every int32 coordinate, score and count is exact there), at
    most DUMP_BYTES in all. An array larger than its share of what is left keeps a sample of its rows drawn with a fixed
    seed, in their original order, so two builds run with the same arguments write comparable files."""
    os.makedirs(out_dir, exist_ok=True)
    budget = DUMP_BYTES - 4096 * len(arrays)                 # room for the .npy headers
    items = sorted(((k, np.asarray(v, dtype=np.float64)) for k, v in arrays.items()), key=lambda kv: kv[1].nbytes)
    for i, (name, a) in enumerate(items):
        share = budget // (len(items) - i)
        if a.nbytes > share:
            keep = share // (a.nbytes // len(a))
            a = a[np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))]
        np.save(os.path.join(out_dir, name + '.npy'), a)
        budget -= a.nbytes


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-lms', '100'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
            # nvidia-smi attaches to the driver while it starts up, which stalls this process's CUDA calls for a while: let
            # it reach its steady 100 ms polling (first row printed) BEFORE the timed region begins, not inside it
            t0 = time.perf_counter()
            while not self.rows and self.proc.poll() is None and time.perf_counter() - t0 < 10.0:
                time.sleep(0.01)
            self.rows_before = len(self.rows)
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(',')])

    def stop(self):
        if not self.proc:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm = [float(r[0]) for r in self.rows if r and r[0].replace('.', '').isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith('active')})
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': reasons, 'samples': len(sm)}


# ------------------------------------------------------------------------------------------------- workloads
class CoverageWorkload:
    """BASELINE config 2: coverage/threshold stage only, 10 M-hit table over a 100 Mbp genome (50 scaffolds x 2 Mbp),
    minCov 3, minLen 100. Under N ranks every rank owns its own 50-scaffold group (weak scaling, no collective)."""
    name = 'C2: coverage/threshold stage, 10M-hit tab over 100 Mbp (50 x 2 Mbp), minCov 3, minLen 100'
    NCHROM, CHROM_SIZE, NHITS, HOTSPOTS = 50, 2_000_000, 10_000_000, 2000
    MIN_COV, MIN_LEN = 3, 100
    dtype = 'int32'

    def __init__(self, rank):
        from tests.helpers import synth_hits
        self.chrom, self.start, self.end, self.sizes = synth_hits(1002 + rank, self.NCHROM, self.CHROM_SIZE, self.NHITS, self.HOTSPOTS)
        self.mbp = self.NCHROM * self.CHROM_SIZE / 1e6

    def to_device(self, torch, dev):
        self.pinned = [torch.from_numpy(a).pin_memory() for a in (self.chrom, self.start, self.end)]
        self.dev = [t.to(dev) for t in self.pinned]
        self.h2d_bytes = sum(t.numel() * 4 for t in self.pinned)

    def step_resident(self):
        from mimeo_b200 import coverage
        out = coverage.coverage_segments_device(self.dev[0], self.dev[1], self.dev[2], self.sizes, self.MIN_COV, self.MIN_LEN)
        self.nseg = int(out[0].numel())
        return out

    def outputs(self, out):
        """What a caller of step_resident receives: the (scaffold, start, end) segments as one [n, 3] array."""
        return {'segments': np.stack([t.cpu().numpy() for t in out], axis=1)}

    def step_e2e(self):
        from mimeo_b200 import coverage
        out = coverage.coverage_segments(self.pinned[0].numpy(), self.pinned[1].numpy(), self.pinned[2].numpy(),
                                         self.sizes, self.MIN_COV, self.MIN_LEN)
        self.d2h_bytes = sum(a.nbytes for a in out)
        self.last_e2e = out
        return out

    def kernel_bytes(self):
        """Algorithmic bytes per launch group (DESIGN.md 'roofline'): H hits, R segments."""
        H, R = self.NHITS, self.nseg
        G = int(self.sizes.sum())
        return {
            'cov_events': 12 * H + 8 * H,                       # read (chrom,start,end), write two event keys
            'cov_bin_events': 2 * 2 * (4 + 4 + 4) * H,          # 2 arrays x 2 radix passes x (hist read + scatter read + write)
            'cov_tile': 8 * H + 8 * R,                          # read both event arrays once, write flips
            '_stage_survey': 12 * H + 4 * G + 16 * H + 4 * G + 12 * R,   # SURVEY 8(d): dense difference-array model
        }

    def cpu_reference(self, threads):
        """CPU oracle port of the same stage (C restatement of genomecov/merge), full workload."""
        import ctypes
        subprocess.check_call(['make', '-C', os.path.join(ROOT, 'oracle'), 'all'], stdout=subprocess.DEVNULL)
        lib = ctypes.CDLL(os.path.join(ROOT, 'oracle', '_build', 'libannot_oracle.so'))
        lib.ora_coverage_segments.restype = ctypes.c_long
        cap = self.NHITS + 8
        oc, os_, oe = (np.zeros(cap, np.int32) for _ in range(3))
        P = lambda a: a.ctypes.data_as(ctypes.c_void_p)
        t0 = time.perf_counter()
        k = lib.ora_coverage_segments(P(self.chrom), P(self.start), P(self.end), ctypes.c_long(self.NHITS), P(self.sizes),
                                      ctypes.c_int(self.NCHROM), ctypes.c_int(self.MIN_COV), ctypes.c_int(self.MIN_LEN),
                                      P(oc), P(os_), P(oe), ctypes.c_long(cap))
        dt = time.perf_counter() - t0
        assert k >= 0
        self.oracle_segments = (oc[:k].copy(), os_[:k].copy(), oe[:k].copy())
        return dt, 1, 'full workload (10M hits / 100 Mbp), arrays already parsed; single-threaded C port of genomecov+merge'

    def parity(self):
        """Segments of the last e2e step vs the C oracle's, element for element (full config-2 size)."""
        got = self.last_e2e
        ok = all(np.array_equal(np.asarray(g), w) for g, w in zip(got, self.oracle_segments))
        return {'segments_identical': bool(ok), 'segments_compared': int(len(self.oracle_segments[0])),
                'scope': 'every (scaffold, start, end) segment of the full 10 M-hit table, GPU vs the C restatement of genomecov+merge'}



def _oracle_pair_job(args):
    """One (target, query) scaffold pair through the CPU LASTZ-restatement (both strands) -- runs in a worker process.
    Returns (seconds, rows in mb2_align's row format with the given ids, oracle stage counters)."""
    ti, tcodes, qi, qcodes, hspthresh = args
    from oracle import lastz_oracle as lo
    st = lo.Stats()
    t0 = time.perf_counter()
    tix = lo.TargetIndex(tcodes)          # LASTZ rebuilds its seed table for every pair: that cost belongs to the baseline
    p = lo.default_params(hspthresh)
    rows = []
    m = len(qcodes)
    for strand, q in ((0, qcodes), (1, lo.revcomp_codes(qcodes))):
        for (s1, e1, s2, e2, sc, nm, nc, _a, _b) in lo.align_tile(tix, q, p, st).tolist():
            qs, qe = (s2 + 1, e2) if strand == 0 else (m - e2 + 1, m - s2)
            rows.append((ti, qi, strand, s1 + 1, e1, qs, qe, sc, nm, nc))
    return time.perf_counter() - t0, rows, st.as_dict()


class AlignWorkload:
    """A `mimeo self / x / map` job on ONE pair of genomes, the pair grid cut into one (target group x query group) block per
    rank (mimeo_b200.parallel.ShardPlan; strong scaling). Per step every rank aligns its block, filters, all-gathers the hit
    table over NCCL, thresholds the coverage of the target scaffolds it owns and sends its segments to rank 0."""
    dtype = 'int32'
    scaling = 'strong'
    mode = 'self'
    MIN_IDT, MIN_LEN, MIN_COV, INTRA_COV, HSPTHRESH, STRICT = 80, 100, 3, 4, 3000, True

    # ---- subclasses provide genomes(): (tnames, tseqs, qnames, qseqs) with tnames in C-locale order; q* is t* for self
    def __init__(self, rank):
        self.tnames, self.tseqs, self.qnames, self.qseqs = self.genomes()
        self.same = self.qseqs is self.tseqs
        self.tsizes = [len(x) for x in self.tseqs]
        self.qsizes = [len(x) for x in self.qseqs]
        self.mbp = (sum(self.tsizes) + (0 if self.same else sum(self.qsizes))) / 1e6
        self.stats = {}
        self.keep_raw = False        # parity leg: also keep the unfiltered rows of the last step

    def covs(self):
        if self.mode == 'map':
            return []
        if self.mode == 'self' and self.STRICT:
            return [('inter', self.MIN_COV), ('intra', self.INTRA_COV)]
        return [('inter', self.MIN_COV)]

    def to_device(self, torch, dev):
        import torch.distributed as dist
        from mimeo_b200 import parallel
        from mimeo_b200.genome import Genome
        self.world = dist.get_world_size() if dist.is_initialized() else 1
        self.rank = dist.get_rank() if dist.is_initialized() else 0
        self.plan = parallel.ShardPlan(self.tsizes, self.qsizes, self.world)
        self.t_idx, self.q_idx = self.plan.block(self.rank)
        self.pinned_t = [torch.from_numpy(np.ascontiguousarray(self.tseqs[i])).pin_memory() for i in self.t_idx]
        share = self.same and self.t_idx == self.q_idx
        self.pinned_q = self.pinned_t if share else [torch.from_numpy(np.ascontiguousarray(self.qseqs[i])).pin_memory() for i in self.q_idx]
        self.T = Genome([self.tnames[i] for i in self.t_idx], [t.numpy() for t in self.pinned_t])
        self.Q = self.T if share else Genome([self.qnames[i] for i in self.q_idx], [t.numpy() for t in self.pinned_q])
        self.Qb = self.Q.both_strands()
        self.hint = None
        if self.same and not share:
            pos = {g: k for k, g in enumerate(self.q_idx)}
            self.hint = [pos.get(g, -1) for g in self.t_idx]
        self.h2d_bytes = sum(self.tsizes[i] for i in self.t_idx) + (0 if share else sum(self.qsizes[i] for i in self.q_idx))
        self.d2h_bytes = 0

    def _annotate(self, hits):
        """hits: rows of this rank's block, already filtered and sorted on the device."""
        from mimeo_b200 import coverage, parallel
        keep_all = lambda h, minLen, minIdt: np.ones(len(h['t_id']), dtype=bool)
        out = parallel.annotate_block(hits, self.t_idx, self.q_idx, self.plan, self.tsizes, self.MIN_IDT, self.MIN_LEN,
                                      coverage.coverage_segments, self.covs(), keep_all, strict_self=(self.mode == 'self' and self.STRICT))
        if out is not None:
            self.table, self.segs = out
            self.nhits, self.nseg = len(self.table), sum(len(v) for v in self.segs.values())
        return out

    def _align_filter(self, T, Q, Qb):
        """alignment + device-side filter / compaction / sort (`mb2_filter_sort`); only the surviving rows cross PCIe."""
        from mimeo_b200 import align as A
        from mimeo_b200.genome import align_params
        dh = A.align_device(T, Q, align_params(self.HSPTHRESH), Q_aux=Qb, t_same_q=self.hint)
        try:
            if self.keep_raw:
                self.raw_hits, _ = dh.download()
            dh.filter_sort(self.MIN_LEN, self.MIN_IDT, map_rule=(self.mode == 'map'))
            hits, self.stats = dh.download()
        finally:
            dh.close()
        return hits

    def step_resident(self):
        return self._annotate(self._align_filter(self.T, self.Q, self.Qb))

    def outputs(self, out):
        """What a caller of step_resident receives on rank 0: the filtered hit table [n, 10] (columns HIT_FIELDS, global
        scaffold ids) and the segments [m, 3] of every coverage pass."""
        if out is None:
            return {}
        table, segs = out
        return {'hits': table, **{f'segments_{name}': v for name, v in segs.items()}}

    def step_e2e(self):
        """Host ASCII (pinned) in -> .tab rows and GFF3 rows out on rank 0, every copy and the collectives inside."""
        from mimeo_b200 import align as A, engine
        from mimeo_b200.genome import Genome
        share = self.pinned_q is self.pinned_t
        T = Genome([self.tnames[i] for i in self.t_idx], [t.numpy() for t in self.pinned_t])
        Q = T if share else Genome([self.qnames[i] for i in self.q_idx], [t.numpy() for t in self.pinned_q])
        try:
            hits = self._align_filter(T, Q, None)
        finally:
            if Q is not T:
                Q.close()
            T.close()
        out = self._annotate(hits)
        if out is None:
            return None
        table, segs = out
        cols = {f: np.ascontiguousarray(table[:, k]) for k, f in enumerate(A.HIT_FIELDS)}
        blocks = A.tab_blocks(cols, self.tnames, self.qnames, 0, 0) if len(table) else {}      # already filtered: format only
        ntab = sum(len(v) for v in blocks.values())
        src = {'self': 'mimeo-self', 'x': 'mimeo', 'map': 'mimeo-map'}[self.mode]
        gff = ''.join(engine.segment_gff_text(v[:, 0], v[:, 1], v[:, 2], self.tnames, src, 'Repeat', 'Repeat') for v in segs.values())
        self.d2h_bytes = 40 * len(table) + 12 * self.nseg
        return ntab, gff.count('\n')

    def kernel_bytes(self):
        """Algorithmic bytes of the HBM-bound seeding kernels per launch (SURVEY 8(d)); one seed_scan launch covers BOTH
        strands of a query chunk, so every term counts both strands."""
        T = sum(self.tsizes[i] for i in self.t_idx)
        Q2 = 2 * sum(self.qsizes[i] for i in self.q_idx)
        S, S_out = self.stats['seed_hits'], self.stats['survivors']
        return {
            'seed_table_build': T // 4 * 2 + 4 * T + 2 * 4 * (1 << 24),
            'seed_scan': Q2 // 4 + Q2 * 13 * 4 + 4 * S + 8 * S_out,          # summed over the launches of a step
        }

    def int_cells(self):
        return {'seed_scan': self.stats['stage1_cells'], 'hsp_extend': self.stats['stage2_cells'], 'gapped': self.stats['gapped_cells']}

    # ---- CPU side
    def sample_pairs(self, npairs):
        """Deterministic sample of the ordered (target, query) scaffold pairs; in self mode every n-th sampled pair is a
        self pair, like the full schedule (n of n*n)."""
        nt, nq = len(self.tnames), len(self.qnames)
        if npairs >= nt * nq:
            return [(a, b) for a in range(nt) for b in range(nq)]
        rng = np.random.default_rng(7)
        flat = rng.choice(nt * nq, size=npairs, replace=False)
        pairs = [(int(f // nq), int(f % nq)) for f in flat]
        if self.mode == 'map':       # scaffold i of B descends from scaffold i of A: a third of the sample are such pairs
            nd = max(1, npairs // 3)
            pairs = [(int(a), int(a)) for a in rng.choice(min(nt, nq), size=min(nd, nt, nq), replace=False)] + [(a, b) for a, b in pairs if a != b][:npairs - nd]
        if self.same:
            nself = max(1, round(npairs / nt))
            pairs = [(a, a) for a in rng.choice(nt, size=min(nself, nt), replace=False).tolist()] + [(a, b) for a, b in pairs if a != b][:npairs - nself]
        return pairs

    def cpu_reference(self, threads, npairs=None, want_rows=False):
        """The CPU LASTZ-restatement on a bounded sample of the job's scaffold pairs, one oracle process per pair on `threads`
        processes (the reference runs one LASTZ process per pair, serially). Returns (wall seconds of the sample, threads,
        description, fraction of the pair grid's area covered, rows or None, oracle gapped cells)."""
        from concurrent.futures import ProcessPoolExecutor
        from oracle import lastz_oracle as lo
        if npairs is None:
            npairs = max(2, 2 * threads)
        pairs = self.sample_pairs(npairs)
        tenc = {a: lo.encode(self.tseqs[a]) for a in {a for a, _ in pairs}}
        qenc = tenc if self.same else {}
        for _, b in pairs:
            if b not in qenc:
                qenc[b] = lo.encode(self.qseqs[b])
        jobs = [(a, tenc[a], b, qenc[b], self.HSPTHRESH) for a, b in pairs]
        t0 = time.perf_counter()
        if threads > 1:
            with ProcessPoolExecutor(max_workers=threads) as ex:
                res = list(ex.map(_oracle_pair_job, jobs, chunksize=1))
        else:
            res = [_oracle_pair_job(j) for j in jobs]
        wall = time.perf_counter() - t0
        area = sum(float(self.tsizes[a]) * float(self.qsizes[b]) for a, b in pairs)
        frac = area / (float(sum(self.tsizes)) * float(sum(self.qsizes)))
        core_s = sum(r[0] for r in res)
        cells = sum(r[2]['gapped_cells'] for r in res)
        sample = (f'{len(pairs)} of {len(self.tnames) * len(self.qnames)} ordered scaffold pairs ({100 * frac:.2f}% of the pair grid by area) '
                  f'through the C LASTZ-restatement incl. per-pair seed-table build, both strands, {threads} process(es): {wall:.1f} s wall, '
                  f'{core_s:.1f} core-seconds; value = job Mbp x sampled fraction / wall')
        rows = None
        if want_rows:
            rows = set()
            for r in res:
                rows.update(r[1])
        return wall, threads, sample, frac, rows, pairs, cells

    def parity(self, oracle_rows, pairs):
        """Rows of the sampled pairs, GPU (last resident step, before filtering) vs oracle."""
        from mimeo_b200.align import HIT_FIELDS
        h = self.raw_hits
        t = np.asarray(self.t_idx, dtype=np.int64)[h['t_id']] if len(h['t_id']) else h['t_id']
        q = np.asarray(self.q_idx, dtype=np.int64)[h['q_id']] if len(h['q_id']) else h['q_id']
        want_pairs = set(pairs)
        got = {(int(t[k]), int(q[k])) + tuple(int(h[f][k]) for f in HIT_FIELDS[2:]) for k in range(len(t)) if (int(t[k]), int(q[k])) in want_pairs}
        return got == oracle_rows, len(oracle_rows)


class SelfWorkload(AlignWorkload):
    """BASELINE config 1: `mimeo self` on a synthetic 5 Mbp genome (10 scaffolds x 500 kbp, 20 planted repeat families of
    5-30 copies at ~80 % pairwise identity), minIdt 80, minLen 100, minCov 3, intraCov 4, --strictSelf."""
    name = 'C1: mimeo self, synthetic 5 Mbp genome (10 x 500 kbp, 20 repeat families at ~80% identity), minIdt 80 minLen 100 minCov 3 intraCov 4 strictSelf'
    mode = 'self'
    NSCAF, SCAF_LEN, NFAM = 10, 500_000, 20

    def genomes(self):
        from tests.helpers import synth_genome
        g = synth_genome(1001, self.NSCAF, self.SCAF_LEN, self.NFAM, copies=(5, 30), fam_len=(300, 3000), sub=0.106, indel=0.005)
        names = sorted(g, key=lambda s: s.encode())
        seqs = [g[n] for n in names]
        self.names, self.seqs, self.sizes = names, seqs, [len(x) for x in seqs]
        return names, seqs, names, seqs


class XWorkload(AlignWorkload):
    """BASELINE config 4: `mimeo x`, genome A 50 Mbp (50 x 1 Mbp) annotated by its hits against genome B 100 Mbp (100 x 1 Mbp),
    40 repeat families 5-30x in B and 1-3x in A at 80-90 % identity, minIdt 80, minLen 100, minCov 5."""
    name = ('C4: mimeo x, synthetic genome A 50 Mbp (50 x 1 Mbp) vs genome B 100 Mbp (100 x 1 Mbp), 40 repeat families (5-30 copies in B, '
            '1-3 in A, 80-90% identity), minIdt 80 minLen 100 minCov 5; Mbp = bases of both genomes')
    mode = 'x'
    MIN_COV = 5

    def genomes(self):
        from tests.helpers import synth_c4
        a, b = synth_c4(1004)
        an, bn = sorted(a, key=lambda s: s.encode()), sorted(b, key=lambda s: s.encode())
        return an, [a[n] for n in an], bn, [b[n] for n in bn]


class MapWorkload(AlignWorkload):
    """BASELINE config 3: `mimeo map`, two 40 Mbp genomes (B = A diverged by 8 % substitutions + 0.5 % indels over 60 % of its
    length, 10 % of the blocks inverted), minIdt 90, minLen 100, no coverage filter."""
    name = ('C3: mimeo map, synthetic genome A 40 Mbp (40 x 1 Mbp) vs B = A diverged (8% substitutions, 0.5% indels over 60% of its length, '
            '10% of blocks inverted), minIdt 90 minLen 100, no coverage filter; Mbp = bases of both genomes')
    mode = 'map'
    MIN_IDT = 90

    def genomes(self):
        from tests.helpers import synth_c3
        a, b = synth_c3(1003)
        an, bn = sorted(a, key=lambda s: s.encode()), sorted(b, key=lambda s: s.encode())
        return an, [a[n] for n in an], bn, [b[n] for n in bn]


class C5Workload(AlignWorkload):
    """BASELINE config 5: `mimeo self` on a 1 Gbp synthetic plant-like genome (40 % repeats, 500 scaffolds). MB2_C5_MBP scales
    the genome down for trial runs (the workload name then says so)."""
    mode = 'self'

    def genomes(self):
        from tests.helpers import synth_c5
        mbp = float(os.environ.get('MB2_C5_MBP', '1000'))
        nscaf = max(8, int(round(500 * mbp / 1000.0)))
        g = synth_c5(1005, int(mbp * 1e6), nscaf)
        names = sorted(g, key=lambda s: s.encode())
        seqs = [g[n] for n in names]
        self.name = ('C5: mimeo self, synthetic plant-like genome %.0f Mbp, %d scaffolds (log-normal lengths), 40%% repeats (families of '
                     '2-10 kbp, 50-2000 copies, 75-98%% identity), minIdt 80 minLen 100 minCov 3 intraCov 4 strictSelf'
                     % (sum(len(x) for x in seqs) / 1e6, nscaf)) + ('' if mbp == 1000 else ' [SCALED-DOWN TRIAL of the 1 Gbp config]')
        return names, seqs, names, seqs


WORKLOADS = {'x': XWorkload, 'self': SelfWorkload, 'map': MapWorkload, 'cov': CoverageWorkload, 'c5': C5Workload}
METRIC = 'self-alignment Mbp/sec (genome Mbp annotated per second of hot-path time)'


# ------------------------------------------------------------------------------------------------- arms
def run_reference(args):
    """The reference's CPU path for this job on the box's host cores: the C LASTZ-restatement (no LASTZ binary exists in the
    image), one process per scaffold pair on every core, each step a bounded sample of the job's pair grid. ms_per_step is
    the measured wall time of a step; value scales the job's Mbp by the sampled fraction of the grid."""
    rank, _, world = env_rank()
    if rank != 0:
        return
    wl = WORKLOADS[args.workload](0)
    cores = os.cpu_count() or 1
    times, frac, sample = [], 1.0, ''
    for i in range(args.warmup + args.steps):
        if args.workload == 'cov':
            dt, used, sample = wl.cpu_reference(cores)
        else:
            dt, used, sample, frac, _, _, _ = wl.cpu_reference(cores, npairs=args.ref_pairs or None)
        if i >= args.warmup:
            times.append(dt)
    ms = 1e3 * float(np.mean(times))
    val = wl.mbp * frac / (ms / 1e3)
    print(json.dumps({
        'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': 'Mbp/s', 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': ms, 'higher_is_better': True, 'scaling': getattr(wl, 'scaling', 'weak'), 'vs_baseline': None, 'dtype': wl.dtype,
        'data': 'synthetic', 'config': {'workload': wl.name},
        'cpu_baseline': {'value': val, 'unit': 'Mbp/s', 'cores': used, 'kind': 'port', 'sample': sample, 'sample_fraction': frac,
                         'host_cpu_count': cores},
        'e2e': {'value': val, 'unit': 'Mbp/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }))


def side_config(workload, steps=5, warmup=3, timeout=900):
    """Another BASELINE config measured by this same script in a fresh process: same arms, same timing rules as the headline;
    the parent holds the GPU idle meanwhile. Returns the child's line, trimmed."""
    env = dict(os.environ, MB2_BENCH_NO_SIDE='1')
    for k in ('RANK', 'LOCAL_RANK', 'WORLD_SIZE'):
        env.pop(k, None)
    out = subprocess.run([sys.executable, os.path.abspath(__file__), '--workload', workload, '--steps', str(steps), '--warmup', str(warmup)],
                         env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=timeout)
    if out.returncode != 0:
        raise RuntimeError(f'child exited {out.returncode}: {out.stderr[-200:]}')
    d = json.loads(out.stdout.strip().splitlines()[-1])
    keep = ('value', 'unit', 'ms_per_step', 'steps', 'warmup', 'e2e', 'gpu_launches', 'clocks', 'cpu_baseline', 'roofline', 'gcups', 'parity')
    r = {k: d[k] for k in keep if k in d}
    r['workload'] = d['config']['workload']
    return r


def run_b200(args):
    import torch
    import torch.distributed as dist
    from mimeo_b200 import _lib
    rank, local_rank, world = env_rank()
    # rank 0 prints ONE JSON line: whatever native libraries write to fd 1 meanwhile (NCCL's version banner) goes to stderr
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    _lib.init(local_rank)
    stream = torch.cuda.ExternalStream(_lib.stream_handle(), device=dev)

    wl = WORKLOADS[args.workload](rank)
    wl.to_device(torch, dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def maxreduce(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- resident arm (value)
    for _ in range(args.warmup):
        wl.step_resident()
    sampler = ClockSampler(local_rank)
    _lib.prof_reset(); _lib.prof_enable(True)
    launches0 = _lib.launch_count()
    if rank == 0:
        sampler.start()
    barrier()
    total_ms = 0.0
    for _ in range(args.steps):
        out = None                          # free the previous step's result first: the step reuses its device buffers
        flush.zero_()                       # L2 flush between timed iterations (outside the timed interval)
        barrier()                           # every rank starts the step together: the step contains collectives
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            out = wl.step_resident()
            e1.record(stream)
        e1.synchronize()
        total_ms += e0.elapsed_time(e1)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    launches = _lib.launch_count() - launches0
    _lib.prof_enable(False)
    ms_step = maxreduce(total_ms / args.steps)
    scaling = getattr(wl, 'scaling', 'weak')
    job_mbp = wl.mbp if scaling == 'strong' else world * wl.mbp
    value = job_mbp / (ms_step / 1e3)

    # ---- roofline of the dominant kernel (same timed region, CUDA events on the library stream)
    peak, peak_src = measured_peaks()
    kb = wl.kernel_bytes()
    hbm_tags = [t for t in kb if not t.startswith('_')]
    int_tags = ['hsp_extend', 'gapped'] if hasattr(wl, 'int_cells') else []
    all_tags = hbm_tags + [t for t in ('surv_sort', 'hsp_extend', 'hsp_sort', 'chain', 'gapped', 'gp_forward', 'cov_events', 'cov_bin_events', 'cov_tile') if t not in hbm_tags]
    prof = {t: _lib.prof_get(t) for t in all_tags}
    sm = _lib.lib().mb2_sm_count()
    int_peak = sm * 128 * 1.965e9                                   # INT32 lane-ops/s at max clock
    budget = {'seed_scan': 6, 'hsp_extend': 6, 'gapped': 12}
    cells = wl.int_cells() if hasattr(wl, 'int_cells') else {}

    def hbm_roofline(tag):
        ms, cnt = prof[tag]
        per_launch_ms = ms / max(cnt, 1)
        launches_per_step = cnt / max(args.steps, 1)
        bytes_per_launch = kb[tag] / max(launches_per_step, 1) if tag == 'seed_scan' else kb[tag]
        achieved = bytes_per_launch / (per_launch_ms / 1e3) / 1e9 if per_launch_ms > 0 else 0.0
        traffic, traffic_src = ncu_traffic(args.workload, tag)
        return {'bound': 'hbm', 'kernel': tag, 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak, 'traffic': traffic,
                'traffic_source': traffic_src, 'peak_source': peak_src, 'ms_per_launch': per_launch_ms, 'launches_per_step': launches_per_step,
                'algorithmic_bytes_per_launch': bytes_per_launch}

    def int_roofline(tag):
        ms = prof[tag][0] / args.steps
        g = cells[tag] / (ms / 1e3) / 1e9 if ms > 0 else 0.0
        return {'bound': 'int32 (integer pipe; no tensor cores: not a dense contraction)', 'kernel': tag, 'achieved': g * budget[tag] / 1e3, 'peak': int_peak / 1e12,
                'unit': 'Tera lane-ops/s at %d ops per cell' % budget[tag], 'frac': g * 1e9 * budget[tag] / int_peak, 'traffic': None,
                'gcups': g, 'cells_per_step': cells[tag], 'ms_per_step': ms}

    dom = max(hbm_tags, key=lambda t: prof[t][0])
    roofline = hbm_roofline(dom)                      # `roofline` = the dominant HBM-bound launch group
    top = max(hbm_tags + int_tags, key=lambda t: prof[t][0])
    roofline['dominant_kernel_of_step'] = top
    if int_tags:
        roofline['int_kernel'] = int_roofline(max(int_tags, key=lambda t: prof[t][0]))
    if dom == 'seed_scan' and cells.get('seed_scan'):
        # the scan's lookups are HBM-shaped but its time goes to the fused first-stage x-drop (ncu: ALU pipe and L1 data pipe ~75 % busy, DRAM 11 %):
        # the same launch against the integer roofline, 6 lane-ops per scored column (SURVEY 8(d))
        ms = prof['seed_scan'][0] / args.steps
        g = cells['seed_scan'] / (ms / 1e3) / 1e9
        roofline['same_kernel_vs_int_roofline'] = {'gcups': g, 'cells_per_step': cells['seed_scan'], 'frac': g * 1e9 * budget['seed_scan'] / int_peak,
                                                   'ops_per_cell': budget['seed_scan'], 'peak_lane_ops_per_s': int_peak}
        if ncu_pipes(args.workload, 'seed_scan'):
            roofline['same_kernel_vs_int_roofline']['ncu_pipe_utilisation'] = ncu_pipes(args.workload, 'seed_scan')
    roofline['kernels_ms_per_step'] = {t: prof[t][0] / args.steps for t in all_tags if prof[t][1]}
    roofline['note'] = ('the kernel with the largest share of the step; `hbm_kernels` lists the HBM-bound launch groups against the measured copy '
                        'peak, `gcups` the integer-pipe kernels (x-drop, y-drop) against the INT32 issue roofline at the SURVEY op budgets')
    roofline['hbm_kernels'] = {t: {k: v for k, v in hbm_roofline(t).items() if k in ('achieved', 'frac', 'ms_per_launch', 'algorithmic_bytes_per_launch', 'traffic')}
                               for t in hbm_tags if prof[t][1]}
    if '_stage_survey' in kb:
        roofline['stage_survey_model'] = {'bytes': kb['_stage_survey'], 'achieved': kb['_stage_survey'] / (ms_step / 1e3) / 1e9,
                                          'frac': kb['_stage_survey'] / (ms_step / 1e3) / 1e9 / peak}
    extra = {}
    if cells:
        gc = {}
        for t, c in cells.items():
            ms = prof[t][0] / args.steps
            if ms > 0:
                g = c / (ms / 1e3) / 1e9
                gc[t] = {'gcups': g, 'cells_per_step': c, 'ms_per_step': ms, 'frac_of_int_roofline': g * 1e9 * budget[t] / int_peak}
        tot_cells = sum(cells.values())
        tot_ms = sum(prof[t][0] for t in cells) / args.steps
        extra['gcups'] = {'value': tot_cells / (tot_ms / 1e3) / 1e9 if tot_ms > 0 else 0.0, 'unit': 'GCUPS (ungapped + gapped cells / kernel seconds), this rank',
                          'per_kernel': gc, 'int_roofline_ops_per_s': int_peak, 'ops_per_cell_budget': budget}
        extra['stage_counters'] = wl.stats
    if hasattr(wl, 'plan'):
        extra['partition'] = {'grid': f'{wl.plan.gt} target groups x {wl.plan.gq} query groups', 'balance': wl.plan.balance,
                              'collectives_per_step': 'all-gather of the filtered hit table + gather of segments to rank 0 (NCCL)' if world > 1 else 'none (1 rank)',
                              'rows_gathered': getattr(wl, 'nhits', None), 'segments': getattr(wl, 'nseg', None)}

    # ---- end-to-end arm through the host-buffer C ABI (H2D + D2H inside the timed region)
    for _ in range(max(1, args.warmup // 2)):
        wl.step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        wl.step_e2e()
    torch.cuda.synchronize()
    e2e_ms = maxreduce(1e3 * (time.perf_counter() - t0) / args.steps)
    barrier()
    e2e = {'value': job_mbp / (e2e_ms / 1e3), 'unit': 'Mbp/s', 'ms_per_step': e2e_ms,
           'h2d_bytes_per_step': wl.h2d_bytes, 'd2h_bytes_per_step': wl.d2h_bytes}

    # ---- the other single-GPU BASELINE configs beside the headline (default workload, 1 GPU only): extra keys, never mixed into `value`
    if rank == 0 and world == 1 and args.workload == DEFAULT_WORKLOAD and not os.environ.get('MB2_BENCH_NO_SIDE'):
        for key, w in (('config1_self_5Mbp', 'self'), ('config2_coverage_stage', 'cov'), ('config3_map_40Mbp', 'map')):
            try:
                extra[key] = side_config(w, steps=args.steps, warmup=args.warmup)
            except Exception as e:      # the headline line must not depend on these legs
                extra[key] = {'error': f'{type(e).__name__}: {e}'[:300]}

    cpu, parity = None, None
    if rank == 0 and world == 1:
        if args.workload == 'cov':
            dt, cores, sample = wl.cpu_reference(1)
            cpu = {'value': wl.mbp / dt, 'unit': 'Mbp/s', 'cores': cores, 'kind': 'port', 'sample': sample, 'seconds': dt}
            parity = wl.parity()
        else:
            # full pair grid for C1 (every row of the benchmarked job is compared); a bounded sample elsewhere
            ncores = os.cpu_count() or 1
            npairs = len(wl.tnames) * len(wl.qnames) if args.workload == 'self' else 12
            dt, cores, sample, frac, rows, pairs, ocells = wl.cpu_reference(min(ncores, npairs), npairs=npairs, want_rows=True)
            core_s = dt * cores
            cpu = {'value': wl.mbp * frac / core_s, 'unit': 'Mbp/s', 'cores': 1, 'kind': 'port', 'sample': sample + f'; reported for ONE core, the reference\'s own schedule (serial LASTZ processes): {core_s:.1f} core-seconds',
                   'seconds': core_s, 'sample_fraction': frac, 'host_cpu_count': ncores, 'oracle_gapped_cells_in_sample': ocells}
            wl.keep_raw = True
            wl.step_resident()
            wl.keep_raw = False
            ok, nrows = wl.parity(rows, pairs)
            parity = {'rows_identical': bool(ok), 'rows_compared': nrows, 'pairs_compared': len(pairs),
                      'scope': 'every alignment row (t, q, strand, start1, end1, start2+, end2+, score, matches, columns) of the sampled scaffold pairs, GPU vs oracle'}
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, wl.outputs(out))

    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    os.close(saved_stdout)
    if rank == 0:
        print(json.dumps({
            'metric': METRIC, 'value': value, 'unit': 'Mbp/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': scaling, 'vs_baseline': None,
            'dtype': wl.dtype, 'data': 'synthetic',
            'config': {'workload': wl.name, 'l2': 'flushed between timed steps (256 MiB memset, outside the timed interval)',
                       'sharding': ('one job; the (target x query) scaffold pair grid cut into one block per rank; hit tables all-gathered, segments gathered to rank 0 inside the timed step'
                                    if scaling == 'strong' else 'one scaffold group of the batch per rank, no data-path collective')},
            'roofline': roofline, 'cpu_baseline': cpu, 'parity': parity, 'e2e': e2e, 'gpu_launches': int(launches), 'clocks': clocks, **extra,
        }))
    if world > 1:
        dist.destroy_process_group()


DEFAULT_WORKLOAD = 'x'


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument('--ref-pairs', type=int, default=0, help='reference arm: scaffold pairs per step (default 2 x host cores)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help="write what the last timed step returned on rank 0 as DIR/<name>.npy (float64, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes what the GPU path computed; the reference arm keeps no outputs')
    args.warmup = max(args.warmup, 3) if args.impl == 'b200' else args.warmup
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
