"""The bench line the driver reads: contract keys of bench.py's GPU arm (short run, one GPU)."""

import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_gpu_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '400', '--warmup', '3', '--cpu-seconds', '1'],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, out.stdout
    line = json.loads(lines[0])
    for key in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling', 'vs_baseline',
                'dtype', 'data', 'config', 'roofline', 'cpu_baseline', 'e2e', 'clocks', 'gpu_launches'):
        assert key in line, key
    assert line['metric'] == 'relabeled transitions/sec' and line['unit'] == 'transitions/s' and line['n_gpus'] == 1
    assert line['steps'] == 400 and line['warmup'] == 3 and line['scaling'] == 'weak' and line['data'] == 'synthetic'
    assert line['config']['key'] == 'c2' and 'workload' in line['config']
    roof = line['roofline']
    assert roof['bound'] == 'hbm' and roof['unit'] == 'GB/s' and 0.05 < roof['frac'] < 1.05
    assert abs(roof['frac'] - roof['achieved'] / roof['peak']) < 1e-6
    assert line['gpu_launches'] >= 400                       # at least one kernel of ours per timed step
    e2e = line['e2e']
    assert e2e['unit'] == line['unit'] and 0 < e2e['value'] < line['value']       # host buffers: PCIe-bound, below the resident rate
    assert e2e['h2d_bytes_per_step'] > 0 and e2e['d2h_bytes_per_step'] > 0 and e2e['steps'] == line['steps']
    cpu = line['cpu_baseline']
    assert cpu['kind'] == 'port' and cpu['cores'] == 1 and cpu['value'] > 0 and cpu['sample']
    assert set(line['clocks']) >= {'sm_mhz', 'sm_max_mhz', 'reasons'}
    # the timed region is exactly --steps launches (~0.7 ms each on C2), and says so
    assert line['steps_timed'] == line['steps'] and line['timed_region_ms'] >= 200
    assert line['clocks']['samples'] >= 5       # (~125 on most boxes: one NVML poll per 2 ms; some boxes answer NVML in ~20 ms)
    assert 0 < e2e['frac_of_link'] < 1.25 and e2e['link_gbs'] > 1   # (back-to-back copies can edge past the probe's serial copies)
    # every BASELINE.json config rides in the same line
    assert set(line['configs']) == {'c1', 'c2', 'c3', 'c4', 'c5'}
    for key, c in line['configs'].items():
        assert c['value'] > 0 and 0.05 < c['roofline']['frac'] < 1.05 and c['roofline']['kernel'], key
        assert c['e2e']['value'] > 0 and c['cpu_baseline']['value'] > 0, key
        # the same launch at a quarter and a sixteenth of the default size: smaller launches pay more of the fixed cost
        sweep = c['launch_size_sweep']
        assert [s['batches_per_launch'] for s in sweep] == [max(1, c['batches_per_launch'] // 4), max(1, c['batches_per_launch'] // 16)], key
        assert all(0.05 < s['frac'] < 1.05 and s['value'] > 0 for s in sweep), key
    assert line['configs']['c2']['value'] == line['value']



def test_bench_dump_outputs_repeat_from_run_to_run(tmp_path):
    """--dump-outputs DIR: a sample of every key of the last timed step's batch as DIR/<config>.<key>.npy in float32 /
    float64, at most 64 MB in all, and the same arrays from a second run with the same arguments."""
    import numpy as np

    dumps = []
    for run in ('a', 'b'):
        out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--config', 'c4', '--steps', '3', '--warmup', '1',
                              '--no-cpu-baseline', '--no-e2e', '--dump-outputs', str(tmp_path / run)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT, env=dict(os.environ, OGB_BENCH_NO_SWEEP='1'))
        assert out.returncode == 0, out.stderr[-2000:]
        assert json.loads(out.stdout.splitlines()[-1])['steps_timed'] == 3
        dumps.append({f: np.load(tmp_path / run / f) for f in os.listdir(tmp_path / run)})
    a, b = dumps
    assert set(a) == set(b) and {f'c4.{k}.npy' for k in ('observations', 'next_observations', 'value_goals', 'actor_goals',
                                                          'actions', 'masks', 'rewards')} <= set(a)
    assert sum(os.path.getsize(tmp_path / 'a' / f) for f in a) <= 64e6
    assert len({len(v) for v in a.values()}) == 1                    # the same transitions of every key
    for name, v in a.items():
        assert v.dtype in (np.float32, np.float64) and len(v) > 0 and np.array_equal(v, b[name]), name

def test_bench_reference_arm_prints_the_same_config():
    common = ['--steps', '3', '--warmup', '1']
    ref = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', *common], capture_output=True, text=True,
                         timeout=600, cwd=ROOT)
    assert ref.returncode == 0, ref.stderr[-2000:]
    line = json.loads([ln for ln in ref.stdout.splitlines() if ln.strip()][-1])
    assert line['impl'] == 'reference' and line['value'] > 0 and line['steps'] == 3 and line['warmup'] == 1
    assert line['cpu_baseline']['kind'] == 'port' and line['cpu_baseline']['cores'] >= 1
    ours = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--config', 'c2', '--no-cpu-baseline', '--no-e2e', *common],
                          capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert ours.returncode == 0, ours.stderr[-2000:]
    assert json.loads(ours.stdout.splitlines()[-1])['config'] == line['config']          # the driver's same_config check
