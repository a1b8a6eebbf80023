"""BASELINE configs[3] (C4) in both MultivariateT reparameterisations, timed in one process.

Hierarchical linear regression, d = 2048 (G = 65 groups x p = 31, 200 observations per group, data seed 20260118),
MultivariateT(df = 100), AlphaDivergence(alpha = 2), S = 256, RMSProp(0.0005) through `_fused_step`, started at
mu = the generating coefficients and Sigma = 0.01 I -- the problem `bench.py --config c4` times in sqrtm mode.

    python tools/run_c4_cholesky.py [--rounds 3] [--chol-iters 100] [--sqrtm-iters 20] [--out profiles/c4_cholesky.json]

After warm-up, the two modes are timed alternately (CUDA events around whole iterations, so a mode's host work counts
only where the GPU waits for it).  A torch.profiler pass over Cholesky-mode iterations then gives the device time of
each stage, and the two triangular kernels' rates are set against the fp64 matmul peak measured in the same run.
Prints one JSON line and writes it to --out.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

# kernel-name substrings of each Cholesky-mode stage (device time summed over the stage's kernels and copies)
STAGES = {
    'draws': ('philox_chisquare_kernel', 'philox_normal_kernel'),
    'rows': ('mvt_rows_kernel',),
    'triangular_transform': ('mvt_chol_trmm_kernel',),
    'model': ('hier_lik_kernel', 'hier_finish_kernel'),
    'weights': ('mvt_logdiag_kernel', 'mvt_weights_kernel', 'mvt_gmu_kernel', 'Memcpy DtoD'),
    'cotangent': ('mvt_chol_cotangent_kernel',),
    'rmsprop': ('rmsprop_step_kernel',),
}


def gpu_identity():
    """Card name, power limit and max SM clock (read-only query)."""
    out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                         capture_output=True, text=True, check=True).stdout.strip()
    name, power, clock = [s.strip() for s in out.split(',')]
    return {'name': name, 'power_limit': power, 'sm_max_clock': clock}


def c4_problem(vb, torch):
    G, p, n_per = 65, 31, 200
    rs = np.random.RandomState(20260118)
    N = G * n_per
    group = np.repeat(np.arange(G), n_per)
    X = rs.randn(N, p)
    m = rs.randn(p)
    beta = m + 0.5 * rs.randn(G, p)
    y = np.sum(X * beta[group], axis=1) + 0.3 * rs.randn(N)
    model = vb.HierarchicalLinearRegression(X, y, group, G)
    d = model.dim
    vp0 = vb.MultivariateT(d, 100).init_param()
    F = np.zeros((d, d))
    F[np.diag_indices(d)] = 0.5 * np.log(0.01)
    vp0[d:] = F[np.tril_indices(d)]
    vp0[:G * p] = beta.reshape(-1)
    vp0[G * p:G * p + p] = m
    return model, d, N, torch.as_tensor(vp0, device='cuda')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--chol-iters', type=int, default=100)
    ap.add_argument('--sqrtm-iters', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--profile-iters', type=int, default=20)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'c4_cholesky.json'))
    args = ap.parse_args()

    import torch
    import viabel_b200 as vb
    import bench
    if not torch.cuda.is_available():
        raise SystemExit('run_c4_cholesky.py needs a CUDA device')
    torch.cuda.set_device(0)
    ident = gpu_identity()
    S = 256
    model, d, N, vp0 = c4_problem(vb, torch)
    np.random.seed(0)                         # AlphaDivergence draws its per-call seed from numpy's global RNG

    arms = {}
    for mode in ('cholesky', 'sqrtm'):
        approx = vb.MultivariateT(d, 100, seed=bench.DRAW_SEED, reparam=mode)
        arms[mode] = dict(obj=vb.AlphaDivergence(approx, model, S, 2.0), opt=vb.RMSProp(0.0005), vp=vp0.clone(), ms=[])

    def step(arm):
        value, grad = arm['obj'](arm['vp'])
        arm['opt']._fused_step(arm['vp'], grad, False)
        return value

    def timed(arm, iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(iters):
            value = step(arm)
        e1.record()
        torch.cuda.synchronize()
        arm['ms'].append(e0.elapsed_time(e1) / iters)
        arm['value'] = float(value)

    for arm in arms.values():
        for _ in range(args.warmup):
            step(arm)
    torch.cuda.synchronize()
    for _ in range(args.rounds):
        timed(arms['cholesky'], args.chol_iters)
        timed(arms['sqrtm'], args.sqrtm_iters)

    # device time per stage (Cholesky mode), torch.profiler with CUDA activities in a pass of its own
    from torch.profiler import ProfilerActivity, profile
    arm = arms['cholesky']
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.profile_iters):
            step(arm)
        torch.cuda.synchronize()
    kernels = {}
    for e in prof.key_averages():
        t = getattr(e, 'device_time_total', None)
        if t is None:
            t = e.cuda_time_total
        if t > 0:
            kernels[e.key] = kernels.get(e.key, 0.0) + t * 1e-3 / args.profile_iters    # us -> ms per iteration
    stages = {}
    for stage, names in STAGES.items():
        hits = {k: v for k, v in kernels.items() if any(n in k for n in names)}
        if not hits:
            raise SystemExit('no device activity found for stage %r (kernels: %s)' % (stage, sorted(kernels)))
        stages[stage] = sum(hits.values())

    peak = bench.matmul_peak_tflops(torch, torch.float64, False, 4096)
    nb = (d + 63) // 64
    useful = float(S) * d * (d + 1)                           # S d (d + 1): each triangular product
    executed = 2.0 * S * 64 * 64 * nb * (nb + 1) / 2          # whole 64-wide tiles on and below the diagonal
    tri = {}
    for name, stage in (('triangular_transform', 'triangular_transform'), ('cotangent', 'cotangent')):
        ms = stages[stage]
        tri[name] = {'kernel_ms': ms, 'useful_flops': useful, 'executed_flops': executed,
                     'tflops': useful / (ms * 1e-3) / 1e12, 'frac_of_fp64_matmul': useful / (ms * 1e-3) / 1e12 / peak}
    med = {k: float(np.median(a['ms'])) for k, a in arms.items()}
    line = {
        'workload': 'hier-linear d=%d (G=65 p=31, %d obs) MultivariateT(df=100) AlphaDivergence(alpha=2) S=%d + '
                    'RMSProp(0.0005) (BASELINE configs[3])' % (d, N, S),
        'var_param_dim': int(vp0.numel()),
        'gpu': ident,
        'ms_per_iter': {'cholesky': med['cholesky'], 'sqrtm': med['sqrtm']},
        'ms_per_iter_rounds': {k: a['ms'] for k, a in arms.items()},
        'iters_per_round': {'cholesky': args.chol_iters, 'sqrtm': args.sqrtm_iters}, 'rounds': args.rounds,
        'speedup': med['sqrtm'] / med['cholesky'],
        'cholesky_stages_ms': stages,
        'cholesky_stages_note': 'device time per iteration from torch.profiler over %d iterations; the gap to '
                                'ms_per_iter is launch / host time' % args.profile_iters,
        'triangular_kernels': tri,
        'fp64_matmul_peak_tflops': peak,
        'peak_note': 'torch.matmul fp64 4096^3 measured in this run (best of 10, bench.matmul_peak_tflops)',
        'final_value': {k: a['value'] for k, a in arms.items()},
        'finite': all(bool(torch.isfinite(a['vp']).all()) for a in arms.values()),
    }
    print(json.dumps(line))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(line, f, indent=1)
        f.write('\n')


if __name__ == '__main__':
    main()
