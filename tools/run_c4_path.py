"""The path-derivative ExclusiveKL at C4 (BASELINE configs[3]) next to the entropy form, in both MultivariateT modes.

Hierarchical linear regression, d = 2048 (the problem of run_c4_cholesky.py), MultivariateT(df = 100),
ExclusiveKL with S = 256, RMSProp(0.0005) through `_fused_step`, started at mu = the generating coefficients and
Sigma = 0.01 I.

    python tools/run_c4_path.py [--rounds 3] [--chol-iters 100] [--sqrtm-iters 10] [--out profiles/c4_path.json]

After warm-up, the Cholesky mode's entropy-form and path-form iterations are timed alternately, then the sqrtm mode's
(CUDA events around whole iterations).  A torch.profiler pass over Cholesky path-form iterations gives the device time
of each stage, new kernels included, and their rates are set against the fp64 matmul rate measured in the same run.
Prints one JSON line and writes it to --out.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

import numpy as np  # noqa: E402

from run_c4_cholesky import c4_problem, gpu_identity  # noqa: E402

# kernel-name substrings of each Cholesky path-form stage (device time summed over the stage's kernels and copies)
STAGES = {
    'draws': ('philox_chisquare_kernel', 'philox_normal_kernel'),
    'rows': ('mvt_rows_kernel',),
    'triangular_transform': ('mvt_chol_trmm_kernel',),
    'model': ('hier_lik_kernel', 'hier_finish_kernel'),
    'inverse_diagonal_blocks': ('mvt_chol_diaginv_kernel',),
    'inverse_doubling': ('mvt_chol_invlevel_kernel',),
    'solve': ('mvt_chol_solve_kernel',),
    'weights': ('mvt_logdiag_kernel', 'mvt_weights_kernel', 'mvt_gmu_kernel', 'Memcpy DtoD'),
    'cotangent': ('mvt_chol_cotangent_kernel',),
    'rmsprop': ('rmsprop_step_kernel',),
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--chol-iters', type=int, default=100)
    ap.add_argument('--sqrtm-iters', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--profile-iters', type=int, default=20)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'c4_path.json'))
    args = ap.parse_args()

    import torch
    import viabel_b200 as vb
    import bench
    if not torch.cuda.is_available():
        raise SystemExit('run_c4_path.py needs a CUDA device')
    torch.cuda.set_device(0)
    ident = gpu_identity()
    S = 256
    model, d, N, vp0 = c4_problem(vb, torch)

    arms = {}
    for mode in ('cholesky', 'sqrtm'):
        for form in ('entropy', 'path'):
            approx = vb.MultivariateT(d, 100, seed=bench.DRAW_SEED, reparam=mode)
            arms[mode, form] = dict(obj=vb.ExclusiveKL(approx, model, S, use_path_deriv=form == 'path'),
                                    opt=vb.RMSProp(0.0005), vp=vp0.clone(), ms=[])

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
        for key in (('cholesky', 'entropy'), ('cholesky', 'path'), ('sqrtm', 'entropy'), ('sqrtm', 'path')):
            timed(arms[key], args.chol_iters if key[0] == 'cholesky' else args.sqrtm_iters)

    from torch.profiler import ProfilerActivity, profile
    arm = arms['cholesky', 'path']
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
    # useful flops: L^-1 is d^3/3 (the doubling levels; the 64 x 64 diagonal blocks are 2 * 64^3 / 6 each),
    # Zhat L^-1 is S d (d + 1)
    diag_flops = nb * 64.0 ** 3 / 3
    rates = {}
    for name, stage, useful in (('inverse_doubling', 'inverse_doubling', d ** 3 / 3.0 - diag_flops),
                                ('inverse_diagonal_blocks', 'inverse_diagonal_blocks', diag_flops),
                                ('solve', 'solve', float(S) * d * (d + 1))):
        ms = stages[stage]
        rates[name] = {'kernel_ms': ms, 'useful_flops': useful, 'tflops': useful / (ms * 1e-3) / 1e12,
                       'frac_of_fp64_matmul': useful / (ms * 1e-3) / 1e12 / peak}
    med = {'%s_%s' % k: float(np.median(a['ms'])) for k, a in arms.items()}
    line = {
        'workload': 'hier-linear d=%d (G=65 p=31, %d obs) MultivariateT(df=100) ExclusiveKL S=%d + RMSProp(0.0005) '
                    '(BASELINE configs[3] with ExclusiveKL)' % (d, N, S),
        'var_param_dim': int(vp0.numel()),
        'gpu': ident,
        'ms_per_iter': med,
        'ms_per_iter_rounds': {'%s_%s' % k: a['ms'] for k, a in arms.items()},
        'iters_per_round': {'cholesky': args.chol_iters, 'sqrtm': args.sqrtm_iters}, 'rounds': args.rounds,
        'path_over_entropy': {'cholesky': med['cholesky_path'] / med['cholesky_entropy'],
                              'sqrtm': med['sqrtm_path'] / med['sqrtm_entropy']},
        'cholesky_path_stages_ms': stages,
        'stages_note': 'device time per iteration from torch.profiler over %d Cholesky path-form iterations; the gap '
                       'to ms_per_iter is launch / host time' % args.profile_iters,
        'path_kernels': rates,
        'fp64_matmul_peak_tflops': peak,
        'peak_note': 'torch.matmul fp64 4096^3 measured in this run (best of 10, bench.matmul_peak_tflops)',
        'final_value': {'%s_%s' % k: a['value'] for k, a in arms.items()},
        'finite': all(bool(torch.isfinite(a['vp']).all()) for a in arms.values()),
    }
    print(json.dumps(line))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(line, f, indent=1)
        f.write('\n')


if __name__ == '__main__':
    main()
