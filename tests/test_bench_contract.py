"""The bench line contract, checked on the lines committed under profiles/ (CPU only: nothing is measured here).
A change of bench.py that drops or renames a key the driver reads shows up as a failure once new lines are committed.
The last two tests cover `--dump-outputs`, the files that let two builds be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def line(name):
    with open(os.path.join(ROOT, 'profiles', name)) as f:
        return json.loads(f.read().strip().splitlines()[-1])


@pytest.mark.parametrize('name', ['r1_bench_c1_v28.json', 'r1_bench_c2_v27_run1.json', 'r1_bench_c2_v27_run2.json'])
def test_b200_line_has_every_contract_key(name):
    d = line(name)
    for k in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling', 'vs_baseline',
              'dtype', 'data', 'config', 'roofline', 'cpu_baseline', 'e2e', 'gpu_launches', 'clocks'):
        assert k in d, k
    assert d['warmup'] >= 3 and d['steps'] >= 1 and d['higher_is_better'] is True and d['data'] == 'synthetic'
    assert d['vs_baseline'] is None                       # BASELINE.md publishes no number for this metric
    assert 'workload' in d['config'] and 'model' not in d['config']
    r = d['roofline']
    assert r['bound'] in ('hbm', 'tensor') and r['unit'] in ('GB/s', 'TFLOP/s')
    assert r['frac'] == pytest.approx(r['achieved'] / r['peak'])
    assert r['achieved'] == pytest.approx(r['algorithmic_bytes_per_launch'] / (r['ms_per_launch'] / 1e3) / 1e9)
    c = d['cpu_baseline']
    assert c['kind'] in ('reference', 'port') and c['cores'] >= 1 and c['value'] > 0 and c['sample']
    e = d['e2e']
    assert e['value'] > 0 and e['h2d_bytes_per_step'] > 0 and e['d2h_bytes_per_step'] > 0
    assert e['value'] != d['value']                       # the end-to-end arm is its own measurement
    assert d['gpu_launches'] > 0
    assert d['clocks']['sm_mhz'] and not set(d['clocks']['reasons']) & {'hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown'}


def test_default_line_carries_config2_from_a_fresh_process():
    c = line('r1_bench_c1_v28.json')['config2_coverage_stage']
    assert 'error' not in c and c['workload'].startswith('C2')
    assert c['ms_per_step'] > 0 and c['e2e']['h2d_bytes_per_step'] == 120_000_000
    assert c['roofline']['kernel'] == 'cov_bin_events' and c['roofline']['traffic'] > 0


def test_reference_line():
    d = line('r1_bench_reference_v25.json')
    assert d['impl'] == 'reference' and d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['value'] == d['value']
    assert d['e2e'] == {'value': d['value'], 'unit': d['unit'], 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}


def test_dump_outputs_are_float64_capped_and_reproducible(tmp_path):
    import bench
    small = np.array([[0, 17, 230]], dtype=np.int32)
    big = np.arange(10_000_000, dtype=np.int32).reshape(-1, 10)        # 80 MB as float64: only a sample fits
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), {'segments': small, 'hits': big})
    files = sorted(os.listdir(tmp_path / 'a'))
    assert files == ['hits.npy', 'segments.npy']
    assert sum(os.path.getsize(tmp_path / 'a' / f) for f in files) <= 64_000_000
    got = {f: np.load(tmp_path / 'a' / f) for f in files}
    assert all(v.dtype == np.float64 for v in got.values())
    assert np.array_equal(got['segments.npy'], small)
    h = got['hits.npy']
    assert h.shape[1] == 10 and 700_000 < len(h) < 1_000_000
    assert (np.diff(h[:, 0]) > 0).all() and (h[:, 9] == h[:, 0] + 9).all()        # whole rows, in their original order
    assert all(np.array_equal(v, np.load(tmp_path / 'b' / f)) for f, v in got.items())


@pytest.mark.gpu
def test_bench_dumps_what_the_last_timed_step_computed(tmp_path):
    """bench.py --dump-outputs on the coverage workload: the segments of the last timed step equal the C oracle's on the
    same seeded input, and the line reports the number of timed steps it was asked for."""
    import bench
    from oracle import annot_oracle as ao
    from tests.helpers import synth_hits
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--workload', 'cov', '--steps', '2', '--warmup', '3',
                        '--dump-outputs', str(tmp_path)], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d['steps'] == 2 and d['parity']['segments_identical']
    assert os.listdir(tmp_path) == ['segments.npy']
    got = np.load(tmp_path / 'segments.npy')
    W = bench.CoverageWorkload
    chrom, start, end, sizes = synth_hits(1002, W.NCHROM, W.CHROM_SIZE, W.NHITS, W.HOTSPOTS)
    want = np.stack(ao.coverage_segments_c(chrom, start, end, sizes, W.MIN_COV, W.MIN_LEN), axis=1)
    assert got.dtype == np.float64 and len(want) > 0 and np.array_equal(got, want)
