"""bench.py's reference arm runs on the CPU: it times the UNMODIFIED reference's nmrfit.equations.objective from
baseline/_ref (or /root/reference), falling back to the oracle port only where neither exists.  One tiny invocation, and
the JSON line carries the keys the driver reads."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--workload', 'c1',
                          '--steps', '2', '--warmup', '3'], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith('{')]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ('impl', 'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
                'vs_baseline', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
        assert key in d, key
    assert d['impl'] == 'reference' and d['unit'] == 'evals/s' and d['value'] > 0 and d['higher_is_better'] is True
    sys.path.insert(0, ROOT)
    from oracle import ref_loader
    want_kind = 'reference' if ref_loader.reference_root() else 'port'
    assert d['cpu_baseline']['kind'] == want_kind and d['cpu_baseline']['cores'] >= 1 and d['cpu_baseline']['value'] == d['value']
    assert d['e2e'] == {'value': d['value'], 'unit': 'evals/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    assert d['vs_baseline'] is None and 'workload' in d['config']


def test_default_workload_is_the_shape_the_metric_is_quoted_on():
    """BASELINE.json: "Voigt objective evals/s (6 peaks, 4k pts)" - both arms default to that shape and describe it with
    the same config, so the driver's ratio compares like with like."""
    sys.path.insert(0, ROOT)
    import bench
    wl = bench.WORKLOADS['metric']
    assert (wl['P'], wl['N']) == (6, 4096)
    cfg = bench.workload_config('metric', 1)
    assert cfg['n_peaks'] == 6 and cfg['n_points'] == 4096 and cfg['workload'] == wl['title']
    import argparse
    saved = sys.argv
    try:
        sys.argv = ['bench.py']
        captured = {}
        bench.run_b200 = lambda a: captured.setdefault('args', a) and 0
        bench.main()
        assert captured['args'].workload == 'metric' and captured['args'].gpus == 1 and captured['args'].warmup >= 3
    finally:
        sys.argv = saved


def test_reference_arm_under_torchrun_ranks_other_than_zero_do_nothing():
    env = dict(os.environ, RANK='1', WORLD_SIZE='2', LOCAL_RANK='1')
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2'],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ''


@pytest.mark.parametrize('extra', [['--steps', '0'], ['--impl', 'reference', '--dump-outputs', 'out']])
def test_bench_rejects_arguments_it_cannot_honour(extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + extra, capture_output=True, text=True,
                         timeout=120, cwd=ROOT)
    assert out.returncode == 2 and out.stdout == '' and 'error' in out.stderr


@pytest.mark.gpu
@pytest.mark.parametrize('workload', ['metric', 'c3'])
def test_dump_outputs_writes_the_last_generation(workload, tmp_path):
    """--dump-outputs: float64 .npy files, 64 MiB at most (c3's swarm state is larger and is sampled), taken after
    exactly warmup + steps generations."""
    steps, warmup = 2, 3
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--quick', '--workload', workload, '--steps',
                          str(steps), '--warmup', str(warmup), '--dump-outputs', str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert len([l for l in out.stdout.splitlines() if l.startswith('{')]) == 1
    sys.path.insert(0, ROOT)
    import bench
    wl = bench.WORKLOADS[workload]
    B, S, D = wl.get('B', 1), wl['S'], 4 + 3 * wl['P']
    got = {f[:-4]: np.load(str(tmp_path / f)) for f in os.listdir(str(tmp_path))}
    assert sum(os.path.getsize(str(tmp_path / f)) for f in os.listdir(str(tmp_path))) <= 64 << 20
    assert all(a.dtype == np.float64 for a in got.values())
    assert got['best_x'].shape == (B, D) and np.all(got['best_generations'] == warmup + steps)
    assert np.all(got['best_stop'] == 0) and np.all(np.isfinite(got['best_f']))
    rows = B * S
    if 'sample_index' in got:
        rows = got['sample_index'].size
        assert workload == 'c3' and rows < B * S and np.all(np.diff(got['sample_index']) > 0)
    for k in ('x', 'v', 'p'):
        assert got['swarm_' + k].shape == (rows, D)
    assert got['swarm_fx'].shape == got['swarm_fp'].shape == (rows,)
    assert np.all(got['swarm_fp'] <= got['swarm_fx'])               # a personal best is never worse than the position
    assert got['e2e_objective'].size == B * S and np.all(np.isfinite(got['e2e_objective']))
