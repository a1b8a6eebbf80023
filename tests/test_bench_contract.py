"""The bench contract.  The reference arm (numpy oracle on host cores) runs here on a tiny shape and must print
ONE JSON line with the keys a reader of the result expects; the keys of the GPU arm's line are checked on the
committed round-1 lines under profiles/.  On the GPU, --dump-outputs writes the last timed step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import relerr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
             'vs_baseline', 'dtype', 'data', 'config', 'e2e'}


def test_reference_arm_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--n-obs', '4000',
                          '--dim', '16', '--mc', '8', '--steps', '2', '--warmup', '1'],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith('{')]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and BASE_KEYS <= set(d)
    assert d['metric'] == 'elbo_grad_iters_per_sec' and d['unit'] == 'iter/s' and d['higher_is_better'] is True
    assert d['value'] > 0 and d['steps'] == 2 and d['warmup'] == 1
    assert set(d['e2e']) == {'value', 'unit', 'h2d_bytes_per_step', 'd2h_bytes_per_step'}
    assert d['e2e']['h2d_bytes_per_step'] == 0 and d['e2e']['value'] == d['value']
    cb = d['cpu_baseline']
    assert cb['kind'] in ('port', 'reference') and cb['cores'] >= 1 and cb['value'] == d['value'] and cb['sample']
    assert 'workload' in d['config']


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK='1', WORLD_SIZE='2')
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2',
                          '--n-obs', '4000', '--dim', '16', '--mc', '8', '--steps', '1', '--warmup', '0'],
                         capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ''


@pytest.mark.parametrize('extra', [['--steps', '0'], ['--impl', 'reference', '--dump-outputs'],
                                   ['--config', 'c4', '--dump-outputs']])
def test_bench_rejects_bad_arguments(tmp_path, extra):
    if extra[-1] == '--dump-outputs':
        extra = extra + [str(tmp_path / 'dump')]
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + extra,
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 2 and out.stdout == '' and not os.path.exists(tmp_path / 'dump'), out.stderr[-2000:]


def test_reference_arm_time_budget():
    """Without --ref-seconds the reference arm times all --steps steps (test_reference_arm_line); with a budget it
    stops early, after at least 2 steps, and says so in the line."""
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--n-obs', '4000',
                          '--dim', '16', '--mc', '8', '--steps', '5', '--warmup', '1', '--ref-seconds', '0'],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith('{')][-1])
    assert d['steps'] == 2 and '2 of the 5 requested steps timed (time budget 0 s)' in d['cpu_baseline']['sample']


@pytest.mark.gpu
@pytest.mark.parametrize('path, tol', [('f64', 1e-10),
                                       # the tensor-core sweep adds fp32 row sums with shared-memory atomics, whose
                                       # order varies from run to run
                                       ('fast', 1e-6)])
def test_dump_outputs_are_the_last_timed_step(tmp_path, path, tol):
    """--dump-outputs writes the value, gradient and iterate of the last timed step.  The bench runs max(W, 3) warm-up
    steps, 16 graph-capture steps, K burst steps, a settle phase whose length follows the measured rate, and then the
    K timed steps from the state the burst left.  So the dump must equal step max(W, 3) + 16 + 2K of an independent
    FusedStep on the same seeded problem, whatever the settle phase's length was."""
    import torch
    import viabel_b200 as vb
    from viabel_b200.engine import FusedStep
    import bench
    N, d, S, W, K = 20000, 64, 32, 3, 5
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--path', path, '--n-obs', str(N),
                          '--dim', str(d), '--mc', str(S), '--steps', str(K), '--warmup', str(W), '--no-psis',
                          '--no-f64', '--no-cpu-baseline', '--dump-outputs', str(tmp_path)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith('{')][-1])
    assert line['steps'] == K and line['finite'] and line['settle_steps'] > 16 + K
    got = {n: np.load(tmp_path / (n + '.npy')) for n in ('value', 'grad', 'var_param')}

    model, approx, objective = bench.device_problem(torch, vb, N, d, S, path)
    eng = FusedStep(objective, vb.RMSProp(0.01))
    eng.set_param(approx.init_param())
    eng.run(max(W, 3) + 16 + 2 * K, use_graph=False)
    want = {'value': eng.value, 'grad': eng.grad, 'var_param': eng.vp}
    for n, a in got.items():
        b = want[n].cpu().numpy()
        assert a.dtype == np.float64 and a.shape == b.shape and np.all(np.isfinite(a)), n
        assert relerr(a, b) < tol, (n, relerr(a, b))


def test_committed_gpu_lines_have_the_contract_keys():
    for name, gpus in (('bench_r01_1gpu.json', 1), ('bench_r01_8gpu.json', 8)):
        with open(os.path.join(ROOT, 'profiles', name)) as f:
            d = json.loads(f.read())
        assert BASE_KEYS | {'clocks', 'gpu_launches', 'roofline', 'cpu_baseline'} <= set(d)
        assert d['n_gpus'] == gpus and d['gpu_launches'] > 0 and d['warmup'] >= 3
        assert {'bound', 'achieved', 'peak', 'unit', 'frac', 'traffic'} <= set(d['roofline'])
        assert abs(d['roofline']['frac'] - d['roofline']['achieved'] / d['roofline']['peak']) < 1e-9
        assert {'sm_mhz', 'sm_max_mhz', 'reasons'} <= set(d['clocks'])
        assert not {'hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown'} & set(d['clocks']['reasons'])
        if gpus == 1:
            assert {'value', 'unit', 'cores', 'kind', 'sample'} <= set(d['cpu_baseline'])
            assert d['e2e']['value'] != d['value'] and d['e2e']['h2d_bytes_per_step'] > 0
