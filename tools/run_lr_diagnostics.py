"""Streaming vi_diagnostics for the low-rank LRGaussian (csrc/lr_stream.cu), timed at the sizes it is for.

  c5   C5's shape: d = 256, n = 1e8 draws, StudentTTarget(df 10) seeded like tools/run_mvt_diagnostics.c5_problem, an
       LRGaussian proposal near the target (sigma about the target scale, B small) at k = 8 and k = 64; the target is
       fused in the kernel.

    python tools/run_lr_diagnostics.py [--n 100000000] [--out profiles/lr_stream_diagnostics.json]
    python -m torch.distributed.run --nproc-per-node 2 tools/run_lr_diagnostics.py --check

For each k: end-to-end draws/s (host clock around vi_diagnostics(keep_samples=False), ending in a device synchronise,
after a warm-up call) and the streaming kernel's time by CUDA events (vb_lr_target_log_weights_f64 alone over all n
draws, P formed beforehand).  In the same run, for comparison at the same d, n and target: the mean-field kernel
(vb_mf_target_log_weights_f64, MFGaussian at the same mu and sigma) and the Cholesky-mode full-rank kernel
(vb_mvt_target_log_weights_f64 on run_mvt_diagnostics' C5 proposal).  The kernels are timed in alternation, best of
--reps.  Card name and power limit are read in the same command.
--check (several ranks): the draw-sharded report against a single-rank one on rank 0, at n = 2e6, both k.
"""
import argparse
import contextlib
import io
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tools'))

import numpy as np  # noqa: E402

KEYS = ('khat', 'd2', 'W1', 'W2', 'mean_error', 'std_error', 'cov_error', 'log_norm_bound')
KS = (8, 64)


def c5_problem(vb, k):
    """(target, LRGaussian(k), var_param, mean-field var_param at the same mu and sigma)"""
    import bench
    d = 256
    rs = np.random.RandomState(20260119)
    loc, scale = rs.randn(d), np.exp(0.25 * rs.randn(d))
    vp_mf = np.concatenate([loc + 0.05 * rs.randn(d), np.log(scale) + 0.10 + 0.02 * rs.randn(d)])
    B = 0.1 * scale[:, None] * rs.randn(d, k) / np.sqrt(k)
    vp = np.concatenate([vp_mf, B.ravel()])
    return vb.StudentTTarget(loc, scale, 10.0), vb.LRGaussian(d, seed=bench.DRAW_SEED, k=k), vp, vp_mf


def timed(torch, fns, reps):
    """CUDA-event times (ms) of each fn, warmed up, then run in alternation `reps` times"""
    for f in fns.values():
        f()
    times = {name: [] for name in fns}
    for _ in range(reps):
        for name, f in fns.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            f()
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1))
    return times


def kernels(vb, torch, n, reps):
    """the LR kernel at each k, the mean-field and the Cholesky-mode MultivariateT kernels: same d, n and target"""
    from viabel_b200 import _lib
    from viabel_b200.convenience import _lr_projection
    import run_mvt_diagnostics
    lw = torch.empty(n, dtype=torch.float64, device='cuda')
    fns = {}

    def lr_fn(k):
        model, approx, vp, _ = c5_problem(vb, k)
        vpd = torch.as_tensor(vp, device='cuda')
        P = _lr_projection(vpd, approx)
        ws = torch.empty(_lib.lib.vb_lr_target_log_weights_workspace_bytes(256, k), dtype=torch.uint8, device='cuda')
        return lambda: _lib.check(_lib.lib.vb_lr_target_log_weights_f64(
            _lib.ptr(vpd), _lib.ptr(P), n, 0, n, 256, k, approx._seed, 0, 1, _lib.ptr(model.loc), _lib.ptr(model.scale),
            10.0, _lib.ptr(lw), None, _lib.ptr(ws), ws.numel(), _lib.stream()))

    for k in KS:
        fns['lr_k%d' % k] = lr_fn(k)
    model, approx, _, vp_mf = c5_problem(vb, 8)
    mfd = torch.as_tensor(vp_mf, device='cuda')
    fns['mf'] = lambda: _lib.check(_lib.lib.vb_mf_target_log_weights_f64(
        _lib.ptr(mfd), n, 256, 0, 0.0, approx._seed, 0, 0, 1, _lib.ptr(model.loc), _lib.ptr(model.scale), 10.0,
        _lib.ptr(lw), None, _lib.stream()))
    mvt_model, mvt, mvt_vp = run_mvt_diagnostics.c5_problem(vb, 'cholesky')
    mvd = torch.as_tensor(mvt_vp, device='cuda')
    mws = torch.empty(_lib.lib.vb_mvt_target_log_weights_workspace_bytes(256), dtype=torch.uint8, device='cuda')
    fns['mvt_cholesky'] = lambda: _lib.check(_lib.lib.vb_mvt_target_log_weights_f64(
        _lib.ptr(mvd), None, n, 0, n, 256, float(mvt.df), mvt._seed, 0, 1, _lib.ptr(mvt_model.loc),
        _lib.ptr(mvt_model.scale), 10.0, _lib.ptr(lw), None, _lib.ptr(mws), mws.numel(), _lib.stream()))
    return timed(torch, fns, reps)


def end_to_end(vb, torch, k, n):
    model, approx, vp, _ = c5_problem(vb, k)
    with contextlib.redirect_stdout(io.StringIO()):
        vb.vi_diagnostics(vp, model=model, approx=approx, n_samples=min(n, 200000), keep_samples=False)   # warm-up
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rep = vb.vi_diagnostics(vp, model=model, approx=approx, n_samples=n, keep_samples=False)
        torch.cuda.synchronize()
        sec = time.perf_counter() - t0
    return {'run': 'c5', 'k': k, 'n_draws': n, 'dim': approx.dim, 'model': type(model).__name__,
            'end_to_end_seconds': sec, 'end_to_end_draws_per_sec': n / sec,
            'report': {key: float(rep[key]) for key in KEYS if key in rep}}


def check(vb, torch):
    """draw-sharded streaming report against a single-rank one (rank 0), C5 shape at n = 2e6, both k"""
    import torch.distributed as dist
    rank = dist.get_rank()
    solo = dist.new_group([0])
    ok = True
    for k in KS:
        model, approx, vp, _ = c5_problem(vb, k)
        with contextlib.redirect_stdout(io.StringIO()):
            shard = vb.vi_diagnostics(vp, model=model, approx=approx, n_samples=2000000, keep_samples=False)
            if rank == 0:
                _, approx1, _, _ = c5_problem(vb, k)
                one = vb.vi_diagnostics(vp, model=model, approx=approx1, n_samples=2000000, keep_samples=False,
                                        group=solo)
        if rank == 0:
            errs = {key: abs(float(shard[key]) - float(one[key])) / max(abs(float(one[key])), 1e-300)
                    for key in KEYS if key in one}
            ok = ok and all(e < 1e-9 for e in errs.values())
            print(json.dumps({'check': 'k%d' % k, 'world': dist.get_world_size(), 'rel_err': errs}))
    dist.barrier()
    return ok


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--n', type=int, default=100000000)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--check', action='store_true')
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'lr_stream_diagnostics.json'))
    args = ap.parse_args()

    import torch
    import viabel_b200 as vb
    if not torch.cuda.is_available():
        raise SystemExit('run_lr_diagnostics.py needs a CUDA device')
    if args.check:
        import torch.distributed as dist
        dist.init_process_group('nccl')
        torch.cuda.set_device(dist.get_rank() % torch.cuda.device_count())
        ok = check(vb, torch)
        dist.destroy_process_group()
        raise SystemExit(0 if ok else 1)
    torch.cuda.set_device(0)
    from run_c4_cholesky import gpu_identity
    gpu = gpu_identity()
    runs = []
    for k in KS:
        runs.append(end_to_end(vb, torch, k, args.n))
        print(json.dumps(runs[-1]), flush=True)
    times = kernels(vb, torch, args.n, args.reps)
    kern = {name: {'ms_best': min(t), 'ms_all': t, 'draws_per_sec': args.n / (min(t) * 1e-3)} for name, t in times.items()}
    print(json.dumps(kern), flush=True)
    out = {'gpu': gpu, 'n_draws': args.n, 'dim': 256,
           'kernel_note': 'CUDA events around one call over all n draws with the Student-t target fused (no theta out), '
                          'the kernels timed in alternation, best of --reps: lr_k* = vb_lr_target_log_weights_f64 (P '
                          'formed beforehand), mf = vb_mf_target_log_weights_f64 (MFGaussian at the same mu, sigma), '
                          'mvt_cholesky = vb_mvt_target_log_weights_f64 in Cholesky mode on the C5 MultivariateT '
                          'proposal of tools/run_mvt_diagnostics.py',
           'end_to_end_note': 'host clock around vi_diagnostics(keep_samples=False) ending in a device synchronise, '
                              'after a warm-up call at n = 2e5: P, draws, log-weights, PSIS and bounds',
           'kernels': kern, 'runs': runs}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(out, f, indent=1)
    print(json.dumps({'wrote': args.out}))


if __name__ == '__main__':
    main()
