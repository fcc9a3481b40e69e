"""bench.py contract.  CPU: the reference arm (the unmodified numba reference when its modules are present, one process per
core; the oracle C port beside it) prints one JSON line with the agreed keys whose `config` is key-identical to the CUDA
arm's; the committed bench lines of the CUDA arm carry every key of the contract.  GPU: --dump-outputs is reproducible."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..')
BASE_KEYS = ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
             'vs_baseline', 'dtype', 'data', 'config', 'e2e')


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '3',
                          '--warmup', '1'], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in BASE_KEYS:
        assert k in d, k
    assert d['impl'] == 'reference' and d['steps'] == 3 and d['warmup'] >= 3          # W >= 3 is enforced
    assert d['metric'] == json.load(open(os.path.join(ROOT, 'BASELINE.json')))['metric']
    assert d['config']['workload'] == 'cfg3' and d['higher_is_better'] is True       # BASELINE configs[2] is the default
    sys.path.insert(0, ROOT)
    import bench
    assert d['config'] == bench.config_dict('cfg3', 1)               # the same dict the CUDA arm prints (same_config)
    c = d['cpu_baseline']
    from oracle import ref_runner
    assert d['value'] > 0 and c['cores'] >= 1 and c['port_value'] > 0
    assert c['kind'] == ('reference' if ref_runner.available() else 'port')
    assert d['e2e'] == {'value': d['value'], 'unit': d['unit'], 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}


def test_committed_bench_line_has_every_contract_key():
    d = json.load(open(os.path.join(ROOT, 'profiles', 'r1', 'bench_cfg2_final.json')))
    for k in BASE_KEYS + ('clocks', 'gpu_launches', 'roofline', 'cpu_baseline'):
        assert k in d, k
    assert d['n_gpus'] == 1 and d['warmup'] >= 3 and d['scaling'] == 'weak' and d['dtype'] == 'f64'
    assert d['gpu_launches'] == 3 * d['steps']
    assert set(('sm_mhz', 'sm_max_mhz', 'reasons')) <= set(d['clocks'])
    assert not set(d['clocks']['reasons']) & {'hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown'}
    r = d['roofline']
    assert r['bound'] == 'hbm' and r['unit'] == 'GB/s' and abs(r['frac'] - r['achieved'] / r['peak']) < 1e-9
    assert r['traffic'] is None or r['traffic'] > 0
    e = d['e2e']
    assert e['h2d_bytes_per_step'] == 4096 * 2 * 8 and e['d2h_bytes_per_step'] > 4096 * 1080 * 4
    assert 0 < e['value'] < d['value']                       # host copies inside the timed region
    c = d['cpu_baseline']
    assert c['kind'] in ('port', 'reference') and c['cores'] >= 1 and c['value'] > 0 and c['sample']
    assert abs(d['value'] - d['steps'] * 4096 / (d['ms_per_step'] * d['steps'] * 1e-3)) / d['value'] < 1e-6


def test_committed_round2_bench_line():
    """The round-2 line (profiles/r2/bench_cfg3_final.json, `python bench.py` on a B200): default workload cfg3, the other
    BASELINE configs under `workloads`, ncu DRAM traffic filled in, the unmodified numba reference as the CPU baseline."""
    sys.path.insert(0, ROOT)
    import bench
    d = json.load(open(os.path.join(ROOT, 'profiles', 'r2', 'bench_cfg3_final.json')))
    for k in BASE_KEYS + ('clocks', 'gpu_launches', 'roofline', 'cpu_baseline', 'workloads', 'e2e_packed_u24'):
        assert k in d, k
    assert d['config'] == bench.config_dict('cfg3', 1) and d['n_gpus'] == 1 and d['gpu_launches'] == 3 * d['steps']
    assert not set(d['clocks']['reasons']) & {'hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown'}
    r = d['roofline']
    assert abs(r['frac'] - r['achieved'] / r['peak']) < 1e-9 and r['traffic'] and r['traffic'] < 0.2 * r['algorithmic_bytes_per_agent_step'] * 32768
    assert set(d['workloads']) == {'cfg2', 'cfg2x2', 'cfg5_270', 'cfg5_540', 'cfg5_1080', 'cfg5_2160'}
    for w in d['workloads'].values():
        assert w['value'] > 1e7 and 0 < w['e2e']['value'] < w['value'] and 0 < w['roofline']['frac'] < 1
    assert d['workloads']['cfg2x2']['value'] > 1e7                     # the north_star target (>= 1e7 at 4096 x 2)
    e = d['e2e']
    assert e['h2d_bytes_per_step'] == 32768 * 2 * 8 and e['d2h_bytes_per_step'] > 32768 * 1080 * 4 and 0 < e['value'] < d['value']
    assert d['e2e_packed_u24']['d2h_bytes_per_step'] < e['d2h_bytes_per_step'] and d['e2e_packed_u24']['value'] > e['value']
    c = d['cpu_baseline']
    assert c['kind'] == 'reference' and c['cores'] >= 1 and 0 < c['value'] < c['port_value']
    ref = json.load(open(os.path.join(ROOT, 'profiles', 'r2', 'bench_reference_arm_final.json')))
    assert ref['impl'] == 'reference' and ref['config'] == d['config'] and ref['cpu_baseline']['kind'] == 'reference'


@pytest.mark.gpu
def test_dump_outputs_repeat_exactly(tmp_path):
    """--dump-outputs writes the last timed tick's observation (float32 / float64, under 64 MB with the flagship's scan
    block sampled); the same arguments give the same arrays bit for bit, and one more timed step changes them."""
    def run(steps, name):
        out = tmp_path / name
        r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', str(steps), '--warmup', '3', '--no-cpu',
                            '--no-extras', '--dump-outputs', str(out)], capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        d = json.loads([l for l in r.stdout.splitlines() if l.strip()][-1])
        assert d['steps'] == steps and d['gpu_launches'] == 3 * steps
        return {f[:-4]: np.load(out / f) for f in sorted(os.listdir(out))}
    a, b, c = run(3, 'a'), run(3, 'b'), run(4, 'c')
    assert set(a) == {'scans_sample', 'state', 'collisions', 'done', 'lap_times', 'lap_counts'}
    assert sum(v.nbytes for v in a.values()) < 64e6
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert a['state'].shape == (7, 32768) and a['scans_sample'].shape[1] == 1080
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    assert not np.array_equal(a['state'], c['state'])
