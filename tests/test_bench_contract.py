"""The bench JSON line contract, checked on the committed records of the round (profiles/r01_bench_*.json), and the
outputs bench.py --dump-outputs writes (on the host, and one run of the benchmark on the GPU)."""
import glob
import json
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RECORDS = sorted(glob.glob(os.path.join(ROOT, 'profiles', 'r01_bench_n[0-9].json')))


@pytest.mark.parametrize('path', RECORDS, ids=[os.path.basename(p) for p in RECORDS])
def test_committed_bench_record_keeps_the_contract(path):
    d = json.loads(open(path).read().strip().splitlines()[-1])
    base = json.load(open(os.path.join(ROOT, 'BASELINE.json')))
    for key in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
                'vs_baseline', 'dtype', 'data', 'config', 'roofline', 'e2e', 'gpu_launches', 'clocks'):
        assert key in d, key
    assert d['unit'] == 'transitions/s' and d['higher_is_better'] is True and d['scaling'] == 'weak'
    assert d['vs_baseline'] is None                        # BASELINE.md publishes no number for this metric
    assert d['data'] == 'synthetic' and d['dtype'] == 'f32' and 'workload' in d['config'] and 'model' not in d['config']
    assert d['warmup'] >= 3 and d['gpu_launches'] >= d['steps'] > 0
    assert d['n_gpus'] == int(os.path.basename(path)[len('r01_bench_n')])
    r = d['roofline']
    assert r['bound'] == 'hbm' and r['unit'] == 'GB/s' and abs(r['frac'] - r['achieved'] / r['peak']) < 1e-9
    assert 0.5 < r['frac'] < 1.0 and (r['traffic'] is None or r['traffic'] > 0)
    # value is the whole-job aggregate: rows per step over the max-over-ranks step time
    rows = r['algorithmic_bytes'] / 828 if 'algorithmic_bytes' in r else None
    if rows:
        assert abs(d['value'] - d['n_gpus'] * rows / (d['ms_per_step'] * 1e-3)) / d['value'] < 1e-6
    e = d['e2e']
    assert e['unit'] == d['unit'] and e['h2d_bytes_per_step'] > 0 and e['d2h_bytes_per_step'] > 0
    assert 0 < e['value'] < d['value']                     # end to end through the plugin API is never the kernel-only number
    c = d['clocks']
    assert c['sm_mhz'] and c['sm_max_mhz'] and not set(c['reasons']) & {'hw_slowdown', 'hw_thermal_slowdown',
                                                                       'sw_thermal_slowdown'}
    assert c['sm_mhz'] >= 0.9 * c['sm_max_mhz']
    if d['n_gpus'] == 1:
        b = d['cpu_baseline']
        assert b['kind'] == 'port' and b['cores'] >= 1 and b['unit'] == d['unit'] and b['sample']
    assert isinstance(base, dict)


def test_dump_outputs_writes_the_same_seeded_sample_of_every_output(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float32 DIR/<name>.npy per output of the HER step, the same rows of each (checked with small
    host tensors standing in for the device ones), and the full-size dump stays under 64 MB."""
    import numpy as np
    import torch
    import bench
    arm, _, _ = bench.synth_dims()
    cols = dict(arm, td=arm['task_descr'], o_2=arm['o'], r=1)           # sample_device's width of each output
    dims = {k: cols[k] for k in bench.HER_OUTPUTS}
    assert bench.DUMP_ROWS * sum(dims.values()) * 4 <= 64 << 20
    monkeypatch.setattr(bench, 'ROWS_PER_STEP', 1000)
    monkeypatch.setattr(bench, 'DUMP_ROWS', 100)
    rows = torch.arange(1000, dtype=torch.float32)[:, None]
    out = {k: rows * 100 + torch.arange(d, dtype=torch.float32) for k, d in dims.items()}
    out['_keep'] = []
    for d in ('a', 'b'):
        bench.dump_outputs(out, str(tmp_path / d))
    assert sorted(os.listdir(str(tmp_path / 'a'))) == sorted(k + '.npy' for k in dims)
    picked = None
    for k, d in dims.items():
        x = np.load(str(tmp_path / 'a' / (k + '.npy')))
        assert x.dtype == np.float32 and x.shape == (100, d)
        assert np.array_equal(x, np.load(str(tmp_path / 'b' / (k + '.npy'))))
        r = x[:, 0] / 100
        assert picked is None or np.array_equal(r, picked)
        picked = r
    assert len(np.unique(picked)) == 100


@pytest.mark.gpu
def test_bench_dump_is_the_same_in_two_runs(tmp_path):
    """Two runs of bench.py with the same arguments dump the same device outputs of their last timed step."""
    import subprocess
    import sys
    import numpy as np
    import bench
    for d in ('a', 'b'):
        p = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--gpus', '1', '--steps', '1', '--warmup', '0',
                            '--no-sweep', '--no-cpu-baseline', '--dump-outputs', str(tmp_path / d)],
                           capture_output=True, timeout=1200)
        assert p.returncode == 0, p.stderr.decode()[-2000:]
    assert sorted(os.listdir(str(tmp_path / 'a'))) == sorted(k + '.npy' for k in bench.HER_OUTPUTS)
    total = 0
    for k in bench.HER_OUTPUTS:
        x = np.load(str(tmp_path / 'a' / (k + '.npy')))
        assert x.dtype == np.float32 and x.shape[0] == bench.DUMP_ROWS and np.isfinite(x).all(), k
        assert np.array_equal(x, np.load(str(tmp_path / 'b' / (k + '.npy')))), k
        total += x.nbytes
    assert total <= 64 << 20
    assert set(np.unique(np.load(str(tmp_path / 'a' / 'r.npy')))) <= {-1.0, 0.0}
    assert np.array_equal(np.load(str(tmp_path / 'a' / 'td.npy')).sum(1), np.ones(bench.DUMP_ROWS, np.float32))


def test_bench_rejects_a_run_without_timed_steps():
    import subprocess
    import sys
    p = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '0'], capture_output=True)
    assert p.returncode == 2 and b'--steps' in p.stderr


def test_reference_arm_record_keeps_the_contract():
    path = os.path.join(ROOT, 'profiles', 'r01_bench_reference_arm.json')
    if not os.path.exists(path):
        pytest.skip('no reference-arm record committed')
    d = json.loads(open(path).read().strip().splitlines()[-1])
    assert d['impl'] == 'reference' and d['unit'] == 'transitions/s' and d['higher_is_better'] is True
    assert d['e2e'] == {'value': d['value'], 'unit': d['unit'], 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    assert d['cpu_baseline']['kind'] in ('port', 'reference') and d['cpu_baseline']['value'] == d['value']
