"""The fused AlphaDivergence step at C2's shape (N = 1e6, d = 512, S = 256, MFGaussian + RMSProp, alpha = 2) on one GPU.

    python tools/run_alpha_step.py [--iters-fast 300] [--iters-f64 100] [--reps 3] [--out profiles/alpha_step.json]

The problem is bench.py's C2 problem (device_problem, same seeds); the tensor-core path runs on fp16-exact draws, as
bench.py does.  For each sweep path:
1. RMSProp.optimize, host clock around the whole call (it ends in a device synchronise), ms per iteration: the fused
   AlphaDivergence step, the per-iteration loop it replaces (the fused path patched off, as the tests do), and the
   fused ExclusiveKL step, alternated --reps times after one warm-up call of each.
   The fused calls include building the engine and capturing its graphs.
2. Steady state from the same start point, CUDA events around the iterations: graph replays of the fused alpha and
   ExclusiveKL steps, and the per-iteration loop (objective + fused RMSProp kernel) that optimize() runs unfused,
   alternated.
3. In a separate pass, torch.profiler: the alpha step's kernels by name, mean time per step.
Prints one JSON line and writes it to --out, with the GPU's name, power limit and maximum SM clock read in the same
run.  Needs a CUDA device.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = [s.strip() for s in q[0].split(',')]
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters-fast', type=int, default=300)
    ap.add_argument('--iters-f64', type=int, default=100)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--n', type=int, default=1000000)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'alpha_step.json'))
    args = ap.parse_args()

    import torch
    import viabel_b200 as vb
    import viabel_b200.engine as engine
    from bench import device_problem
    from viabel_b200.engine import FusedStep
    torch.cuda.set_device(0)
    N, d, S, alpha = args.n, 512, 256, 2.0
    out = {'gpu': gpu_info(), 'shape': dict(N=N, d=d, S=S, alpha=alpha, family='MFGaussian', optimizer='RMSProp(0.01)'),
           'paths': {}}
    supported = engine.fused_step_supported

    for path, iters in (('fast', args.iters_fast), ('f64', args.iters_f64)):
        model, approx, ekl = device_problem(torch, vb, N, d, S, path)
        alp = vb.AlphaDivergence(approx, model, S, alpha)
        vp0 = approx.init_param()
        assert supported(alp, vb.RMSProp(0.01))

        def optimize(obj, fused):
            engine.fused_step_supported = supported if fused else (lambda *a, **k: False)
            try:
                opt = vb.RMSProp(0.01)
                opt.progress = False
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                res = opt.optimize(iters, obj, vp0)
                sec = time.perf_counter() - t0
            finally:
                engine.fused_step_supported = supported
            assert np.all(np.isfinite(res['value_history']))
            return sec / iters

        arms = {'alpha_fused': lambda: optimize(alp, True), 'alpha_unfused': lambda: optimize(alp, False),
                'exclusive_kl_fused': lambda: optimize(ekl, True)}
        for fn in arms.values():
            fn()                                                       # warm-up: module loads, tensor maps
        times = {k: [] for k in arms}
        for _ in range(args.reps):
            for k, fn in arms.items():
                times[k].append(fn() * 1e3)
        res = {k: dict(ms_per_iter=float(np.median(v)), runs=v) for k, v in times.items()}
        res['unfused_over_fused'] = res['alpha_unfused']['ms_per_iter'] / res['alpha_fused']['ms_per_iter']
        res['alpha_over_exclusive_kl'] = res['alpha_fused']['ms_per_iter'] / res['exclusive_kl_fused']['ms_per_iter']

        # steady state from the same start: graph replays of the fused steps, and the per-iteration loop
        # (objective(vp) + the fused RMSProp kernel, what optimize() runs unfused), CUDA events around `iters` steps
        engs = {}
        for name, obj in (('alpha', alp), ('exclusive_kl', ekl)):
            eng = FusedStep(obj, vb.RMSProp(0.01), hist_len=4 * iters)
            eng.set_param(vp0)
            if eng.alpha:
                eng.set_seeds(0, np.random.RandomState(5).randint(2 ** 32, dtype=np.uint64, size=4 * iters))
            eng.run(16)
            engs[name] = eng
        vpd = torch.as_tensor(vp0, device='cuda')
        vloop = vpd.clone()
        lopt = vb.RMSProp(0.01)

        def loop():
            for _ in range(iters):
                _, g = alp(vloop)
                lopt._fused_step(vloop, g, False)

        def timed(fn):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            fn()
            b.record()
            b.synchronize()
            return a.elapsed_time(b) / iters

        steps = {'alpha_fused': [], 'alpha_unfused': [], 'exclusive_kl_fused': []}
        for _ in range(args.reps):
            for name, eng in engs.items():
                eng.restart()
                eng.set_param(vp0)
                steps[name + '_fused'].append(timed(lambda: eng.run(iters)))
                if name == 'alpha':
                    vloop.copy_(vpd)
                    lopt.reset_state()
                    steps['alpha_unfused'].append(timed(loop))
        res['steady_ms_per_step'] = {k: dict(median=float(np.median(v)), runs=v) for k, v in steps.items()}
        res['steady_unfused_over_fused'] = (res['steady_ms_per_step']['alpha_unfused']['median']
                                            / res['steady_ms_per_step']['alpha_fused']['median'])
        res['launches_per_step'] = {k: e.launches_per_step for k, e in engs.items()}

        # stage breakdown of the alpha step (separate pass, profiler on)
        from torch.profiler import ProfilerActivity, profile
        eng = engs['alpha']
        eng.restart()
        nprof = min(iters, 32)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            eng.run(nprof)
            torch.cuda.synchronize()
        stages = {}
        for ev in prof.key_averages():
            if ev.device_type is not None and 'CUDA' in str(ev.device_type) and ev.count > 0:
                t = getattr(ev, 'device_time_total', None)
                if t is None:
                    t = ev.cuda_time_total
                stages[ev.key] = dict(calls_per_step=ev.count / nprof, us_per_step=t / nprof)
        res['alpha_stages'] = dict(sorted(stages.items(), key=lambda kv: -kv[1]['us_per_step']))
        res['iters'] = iters
        out['paths'][path] = res
        del engs, eng, model, approx, ekl, alp
        torch.cuda.empty_cache()

    out['multi_gpu'] = 'not run: one GPU'
    line = json.dumps(out)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        f.write(json.dumps(out, indent=1) + '\n')


if __name__ == '__main__':
    main()
