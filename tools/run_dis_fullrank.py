"""DISInclusiveKL on the full-rank and low-rank families, timed on one GPU in one process.

    python tools/run_dis_fullrank.py [--iters 40] [--rounds 3] [--out profiles/dis_fullrank.json]

1. DIS + RMSProp(0.0005) on C4's problem (hierarchical linear regression, d = 2048, tools/run_c4_cholesky.py) for
   MultivariateT(df = 100) in both reparameterisations: S = 256, ess_target = 64, num_resampling_batches = 4 (one
   refresh -- draws, model, bisection -- every 4 calls, a resampled batch of 16 rows otherwise), temper prior
   MFGaussian at the start point.  Refresh and non-refresh iterations are timed separately (host clock around each
   iteration, which ends in the objective's own host read of the weights or of the resampling indices).
2. LRGaussian at d = 256, k in {8, 64} on a product Gaussian target, the same DIS settings.
3. torch.profiler device time per stage of the MultivariateT score (inverse, Y, V, cotangent) and of a refresh
   (draws and model, bisection), and the score products' FP64 rate against torch's fp64 matmul measured in this run.
4. The score alone, alternated in one process with a torch-autograd score of the same closed form (triangular solves
   for MultivariateT, Woodbury for LRGaussian) at the shapes above.
Prints one JSON line and writes it to --out.  Needs a CUDA device.
"""
import argparse
import json
import math
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

import numpy as np  # noqa: E402

SCORE_STAGES = {
    'inverse': ('mvt_chol_diaginv_kernel', 'mvt_chol_invlevel_kernel'),
    'Y': ('mvt_chol_trmm_kernel',),
    'rows_value': ('mvt_score_rows_kernel', 'mvt_score_value_kernel', 'mvt_logdiag_kernel'),
    'V': ('mvt_chol_solve_kernel',),
    'gmu': ('mvt_gmu_kernel',),
    'cotangent': ('mvt_chol_cotangent_kernel',),
}
REFRESH_STAGES = {
    'draws_transform': ('philox_', 'mvt_rows_kernel', 'mvt_chol_trmm_kernel'),
    'model': ('hier_',),
    'bisection': ('dis_bisection_kernel',),
}


def torch_mvt_score(torch, vp, x, idx, c, d, df):
    """the same closed form under torch autograd: y = L^-1 (x - mu) by a triangular solve"""
    lam = vp.detach().clone().requires_grad_(True)
    mu = lam[:d]
    ii = torch.tril_indices(d, d, device=vp.device)
    F = torch.zeros(d, d, dtype=vp.dtype, device=vp.device).index_put((ii[0], ii[1]), lam[d:])
    L = torch.tril(F, -1) + torch.diag(torch.exp(torch.diagonal(F)))
    D = (x[idx] - mu).T
    Y = torch.linalg.solve_triangular(L, D, upper=False)
    delta = (Y * Y).sum(dim=0)
    lq = -torch.diagonal(F).sum() - 0.5 * (df + d) * torch.log1p(delta / df)
    value = -(c * lq).sum()
    (g,) = torch.autograd.grad(value, lam)
    return value.detach(), g


def torch_lr_score(torch, vp, x, idx, c, d, k):
    lam = vp.detach().clone().requires_grad_(True)
    mu, ls, B = lam[:d], lam[d:2 * d], lam[2 * d:].reshape(d, k)
    Dinv2 = torch.exp(-2 * ls)
    M = torch.eye(k, dtype=vp.dtype, device=vp.device) + B.T @ (B * Dinv2[:, None])
    diff = x[idx] - mu
    t = (diff * Dinv2) @ B
    maha = (diff * diff * Dinv2).sum(dim=1) - (t * torch.linalg.solve(M, t.T).T).sum(dim=1)
    lq = -0.5 * (2 * ls.sum() + torch.linalg.slogdet(M)[1] + maha)
    value = -(c * lq).sum()
    (g,) = torch.autograd.grad(value, lam)
    return value.detach(), g


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=40)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--score-reps', type=int, default=20)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'dis_fullrank.json'))
    args = ap.parse_args()

    import torch
    import viabel_b200 as vb
    import bench
    from run_c4_cholesky import c4_problem, gpu_identity
    if not torch.cuda.is_available():
        raise SystemExit('run_dis_fullrank.py needs a CUDA device')
    torch.cuda.set_device(0)
    ident = gpu_identity()
    S, ess_target, batches = 256, 64, 4
    out = {'gpu': ident, 'settings': {'S': S, 'ess_target': ess_target, 'num_resampling_batches': batches,
                                      'rmsprop_lr': 0.0005, 'iters_per_round': args.iters, 'rounds': args.rounds}}

    def dis_arm(approx, model, vp0, prior_params):
        obj = vb.DISInclusiveKL(approx, model, S, ess_target, vb.MFGaussian(approx.dim), prior_params,
                                num_resampling_batches=batches)
        return dict(obj=obj, opt=vb.RMSProp(0.0005), vp=vp0.clone(), refresh=[], other=[], error=None)

    def run_arm(arm, iters):
        for _ in range(iters):
            refresh = arm['obj']._objective_step % batches == 0
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            _, grad = arm['obj'](arm['vp'])
            arm['opt']._fused_step(arm['vp'], grad, False)
            torch.cuda.synchronize()
            (arm['refresh'] if refresh else arm['other']).append((time.perf_counter() - t0) * 1e3)

    def summary(arm):
        if arm['error']:
            return {'error': arm['error']}
        return {'refresh_ms': float(np.median(arm['refresh'])), 'non_refresh_ms': float(np.median(arm['other'])),
                'n_refresh': len(arm['refresh']), 'n_non_refresh': len(arm['other']),
                'finite': bool(torch.isfinite(arm['vp']).all())}

    # 1. C4 in both modes
    model, d, N, vp0 = c4_problem(vb, torch)
    prior = torch.cat([vp0[:d], torch.full((d,), 0.5 * math.log(0.01), dtype=torch.float64, device='cuda')])
    np.random.seed(0)
    arms = {mode: dis_arm(vb.MultivariateT(d, 100, seed=bench.DRAW_SEED, reparam=mode), model, vp0, prior)
            for mode in ('cholesky', 'sqrtm')}
    for _ in range(args.rounds + 1):                     # the first round is warm-up
        for arm in arms.values():
            if arm['error'] is None:
                try:
                    run_arm(arm, args.iters if arm['refresh'] or arm['other'] else batches)
                except (ValueError, NotImplementedError) as e:
                    arm['error'] = '%s: %s' % (type(e).__name__, e)
    out['c4_mvt'] = {mode: summary(arm) for mode, arm in arms.items()}
    out['c4_mvt']['workload'] = ('hier-linear d=%d (G=65 p=31, %d obs), MultivariateT(df=100), start at the generating '
                                 'coefficients with Sigma = 0.01 I' % (d, N))

    # 2. LRGaussian, d = 256
    out['lr_d256'] = {}
    for k in (8, 64):
        dl = 256
        mean, sd = np.linspace(-1, 1, dl), np.linspace(0.5, 1.5, dl)
        approx = vb.LRGaussian(dl, seed=3, k=k)
        vpl = torch.as_tensor(np.concatenate([mean, np.log(sd), 0.1 * np.random.RandomState(k).randn(dl * k)]),
                              device='cuda')
        arm = dis_arm(approx, vb.GaussianTarget(mean, sd), vpl,
                      torch.as_tensor(np.concatenate([mean, np.log(2 * sd)]), device='cuda'))
        try:
            run_arm(arm, batches)
            for _ in range(args.rounds):
                run_arm(arm, args.iters)
        except (ValueError, NotImplementedError) as e:
            arm['error'] = '%s: %s' % (type(e).__name__, e)
        out['lr_d256']['k=%d' % k] = summary(arm)

    # 3. stage breakdown of the MultivariateT score and of a refresh (Cholesky mode)
    from torch.profiler import ProfilerActivity, profile
    rs = np.random.RandomState(1)
    xs = torch.as_tensor(rs.randn(S, d) * 0.1, device='cuda') + vp0[:d]
    arm = arms['cholesky']
    n_batch = max(1, ess_target // batches)
    idx = torch.as_tensor(rs.randint(0, S, n_batch), device='cuda')
    obj = arm['obj']

    def kernel_ms(prof, reps):
        ks = {}
        for e in prof.key_averages():
            t = getattr(e, 'device_time_total', None)
            if t is None:
                t = e.cuda_time_total
            if t > 0:
                ks[e.key] = ks.get(e.key, 0.0) + t * 1e-3 / reps
        return ks

    def stages(ks, table):
        return {s: sum(v for k, v in ks.items() if any(n in k for n in names)) for s, names in table.items()}

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.score_reps):
            obj._score(arm['vp'], xs, idx, None, 1.0)
        torch.cuda.synchronize()
    score_stages = stages(kernel_ms(prof, args.score_reps), SCORE_STAGES)
    if arm['error'] is None:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(batches):
                obj(arm['vp'])
            torch.cuda.synchronize()
        refresh_stages = stages(kernel_ms(prof, 1), REFRESH_STAGES)
    else:
        refresh_stages = {'error': arm['error']}
    peak = bench.matmul_peak_tflops(torch, torch.float64, False, 4096)
    nb = (d + 63) // 64
    useful = {'Y': float(n_batch) * d * (d + 1), 'V': float(n_batch) * d * (d + 1),
              'cotangent': float(n_batch) * d * (d + 1), 'inverse': d ** 3 / 3.0}
    out['mvt_score_stages_ms'] = score_stages
    out['mvt_score_rates'] = {s: {'kernel_ms': score_stages[s], 'useful_flops': f,
                                  'tflops': f / (score_stages[s] * 1e-3) / 1e12 if score_stages[s] > 0 else None,
                                  'frac_of_fp64_matmul': (f / (score_stages[s] * 1e-3) / 1e12 / peak
                                                          if score_stages[s] > 0 else None)}
                              for s, f in useful.items()}
    out['mvt_score_note'] = ('score of one resampled batch of %d rows at d = %d; executed tiles are whole 64-wide '
                             'triangles (%d column blocks)' % (n_batch, d, nb))
    out['refresh_stages_ms'] = refresh_stages
    out['fp64_matmul_peak_tflops'] = peak

    # 4. kernel score vs torch autograd of the same closed form, alternated
    def alt(kernel, ref, reps):
        ks, ts = [], []
        kernel()                                         # warm-up of both shapes
        ref()
        for _ in range(args.rounds):
            for fn, acc in ((kernel, ks), (ref, ts)):
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(reps):
                    fn()
                e1.record()
                torch.cuda.synchronize()
                acc.append(e0.elapsed_time(e1) / reps)
        return {'kernel_ms': float(np.median(ks)), 'torch_autograd_ms': float(np.median(ts))}

    out['score_vs_torch'] = {}
    df = 100.0
    for n in (n_batch, S):
        ii = torch.as_tensor(rs.randint(0, S, n), device='cuda')
        c = torch.full((n,), 1.0, dtype=torch.float64, device='cuda')
        out['score_vs_torch']['mvt d=%d n=%d' % (d, n)] = alt(
            lambda: obj._score(arm['vp'], xs, ii, None, 1.0),
            lambda: torch_mvt_score(torch, arm['vp'], xs, ii, c, d, df), args.score_reps)
    for k in (8, 64):
        dl = 256
        approx = vb.LRGaussian(dl, seed=3, k=k)
        vpl = torch.as_tensor(np.concatenate([np.zeros(dl), np.zeros(dl), 0.1 * rs.randn(dl * k)]), device='cuda')
        xl = torch.as_tensor(rs.randn(S, dl), device='cuda')
        objl = vb.DISInclusiveKL(approx, vb.Model(lambda z: -(z ** 2).sum(dim=1)), S, ess_target, vb.MFGaussian(dl),
                                 np.zeros(2 * dl))
        for n in (n_batch, S):
            ii = torch.as_tensor(rs.randint(0, S, n), device='cuda')
            c = torch.full((n,), 1.0, dtype=torch.float64, device='cuda')
            out['score_vs_torch']['lr d=%d k=%d n=%d' % (dl, k, n)] = alt(
                lambda: objl._score(vpl, xl, ii, None, 1.0), lambda: torch_lr_score(torch, vpl, xl, ii, c, dl, k),
                args.score_reps)
    print(json.dumps(out))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(out, f, indent=1)
        f.write('\n')


if __name__ == '__main__':
    main()
