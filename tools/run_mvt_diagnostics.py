"""Streaming vi_diagnostics for the full-rank MultivariateT (csrc/mvt_stream.cu), timed at the sizes it is for.

  c5        C5's shape: d = 256, n = 1e8 draws, StudentTTarget(df 10) seeded like bench.bench_c5, a MultivariateT(df 40)
            proposal at the same point (diagonal Sigma) -- once per reparameterisation; the target is fused in the kernel.
  c4_chol   the C4 problem (hierarchical linear regression, d = 2048, tools/run_c4_cholesky.c4_problem) with n = 1e6
            draws in Cholesky mode: theta leaves the kernel in 2 GB chunks and the model adds log p.

    python tools/run_mvt_diagnostics.py [--n-c5 100000000] [--n-c4 1000000] [--out profiles/mvt_stream_diagnostics.json]
    python -m torch.distributed.run --nproc-per-node 2 tools/run_mvt_diagnostics.py --check

For each run: end-to-end draws/s (host clock around vi_diagnostics(keep_samples=False), ending in a device
synchronise, after a warm-up call), the streaming kernel's time by CUDA events (draws through vb_mvt_target_log_weights_f64
alone, the sqrtm map formed beforehand), and its FP64 rate on algorithmic flops (n d (d + 1) triangular, 2 n d^2 dense)
against torch.matmul fp64 measured in the same run.  Card name and power limit are read in the same command.
--check (several ranks): the draw-sharded report against a single-rank one on rank 0, at n = 2e6.
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


def c5_problem(vb, mode):
    import bench
    d = 256
    rs = np.random.RandomState(20260119)
    loc, scale = rs.randn(d), np.exp(0.25 * rs.randn(d))
    vp_mf = np.concatenate([loc + 0.05 * rs.randn(d), np.log(scale) + 0.10 + 0.02 * rs.randn(d)])
    F = np.diag(vp_mf[d:])
    vp = np.concatenate([vp_mf[:d], F[np.tril_indices(d)]])
    return vb.StudentTTarget(loc, scale, 10.0), vb.MultivariateT(d, 40, seed=bench.DRAW_SEED, reparam=mode), vp


def kernel_ms(vb, torch, vp, model, approx, n, reps):
    """CUDA-event time of the streaming kernel alone over n draws (fused target, or theta_out chunks for a model)."""
    from viabel_b200 import _lib
    from viabel_b200.models import _product_target
    d = approx.dim
    vpd = torch.as_tensor(vp, device='cuda')
    A = None
    if approx.reparam == 'sqrtm':
        _, _, w, V = approx.decompose(vpd)
        A = torch.empty(d, d, dtype=torch.float64, device='cuda')
        _lib.check(_lib.lib.vb_gemm_f64(0, 1, d, d, d, 1.0, _lib.ptr(V), d, _lib.ptr(V), d, _lib.ptr(A), d,
                                        _lib.ptr(torch.sqrt(w)), None, None, None, None, _lib.stream()))
    ws = torch.empty(_lib.lib.vb_mvt_target_log_weights_workspace_bytes(d), dtype=torch.uint8, device='cuda')
    lw = torch.empty(n, dtype=torch.float64, device='cuda')
    target = _product_target(model)
    fused = target is not None
    chunk = n if fused else max(1, 2 ** 28 // d)
    theta = None if fused else torch.empty(min(chunk, n), d, dtype=torch.float64, device='cuda')
    kind, loc, scale, tdf = target if fused else (-1, None, None, 0.0)

    def once():
        for lo in range(0, n, chunk):
            m = min(chunk, n - lo)
            _lib.check(_lib.lib.vb_mvt_target_log_weights_f64(
                _lib.ptr(vpd), _lib.ptr(A), n, lo, m, d, float(approx.df), approx._seed, 0, kind,
                _lib.ptr(loc), _lib.ptr(scale), tdf,
                _lib.ptr(lw[lo:lo + m]), _lib.ptr(None if theta is None else theta[:m]), _lib.ptr(ws), ws.numel(),
                _lib.stream()))
    once()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = []
    for _ in range(reps):
        e0.record()
        once()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    return min(times), times


def run(vb, torch, name, model, approx, vp, n, peak, reps):
    small = min(n, 200000)
    with contextlib.redirect_stdout(io.StringIO()):
        vb.vi_diagnostics(vp, model=model, approx=approx, n_samples=small, keep_samples=False)      # warm-up
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rep = vb.vi_diagnostics(vp, model=model, approx=approx, n_samples=n, keep_samples=False)
        torch.cuda.synchronize()
        sec = time.perf_counter() - t0
    d = approx.dim
    ms, all_ms = kernel_ms(vb, torch, vp, model, approx, n, reps)
    flops = n * d * (d + 1) if approx.reparam == 'cholesky' else 2 * n * d * d
    tflops = flops / (ms * 1e-3) / 1e12
    return {'run': name, 'reparam': approx.reparam, 'n_draws': n, 'dim': d, 'model': type(model).__name__,
            'end_to_end_seconds': sec, 'end_to_end_draws_per_sec': n / sec,
            'kernel_ms_best': ms, 'kernel_ms_all': all_ms, 'kernel_draws_per_sec': n / (ms * 1e-3),
            'algorithmic_flops': flops, 'kernel_fp64_tflops': tflops, 'frac_of_fp64_matmul': tflops / peak,
            'report': {k: float(rep[k]) for k in KEYS if k in rep}}


def check(vb, torch):
    """draw-sharded streaming report against a single-rank one (rank 0), C5 shape at n = 2e6, both modes"""
    import torch.distributed as dist
    rank = dist.get_rank()
    solo = dist.new_group([0])
    ok = True
    for mode in ('cholesky', 'sqrtm'):
        model, approx, vp = c5_problem(vb, mode)
        with contextlib.redirect_stdout(io.StringIO()):
            shard = vb.vi_diagnostics(vp, model=model, approx=approx, n_samples=2000000, keep_samples=False)
            if rank == 0:
                _, approx1, _ = c5_problem(vb, mode)
                one = vb.vi_diagnostics(vp, model=model, approx=approx1, n_samples=2000000, keep_samples=False,
                                        group=solo)
        if rank == 0:
            errs = {k: abs(float(shard[k]) - float(one[k])) / max(abs(float(one[k])), 1e-300) for k in KEYS if k in one}
            ok = ok and all(e < 1e-9 for e in errs.values())
            print(json.dumps({'check': mode, 'world': dist.get_world_size(), 'rel_err': errs}))
    dist.barrier()
    return ok


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--n-c5', type=int, default=100000000)
    ap.add_argument('--n-c4', type=int, default=1000000)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--check', action='store_true')
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'mvt_stream_diagnostics.json'))
    args = ap.parse_args()

    import torch
    import viabel_b200 as vb
    if not torch.cuda.is_available():
        raise SystemExit('run_mvt_diagnostics.py needs a CUDA device')
    if args.check:
        import torch.distributed as dist
        dist.init_process_group('nccl')
        torch.cuda.set_device(dist.get_rank() % torch.cuda.device_count())
        ok = check(vb, torch)
        dist.destroy_process_group()
        raise SystemExit(0 if ok else 1)
    torch.cuda.set_device(0)
    import bench
    from run_c4_cholesky import c4_problem, gpu_identity
    peak = bench.matmul_peak_tflops(torch, torch.float64, False, 4096)
    runs = []
    for mode in ('cholesky', 'sqrtm'):
        model, approx, vp = c5_problem(vb, mode)
        runs.append(run(vb, torch, 'c5', model, approx, vp, args.n_c5, peak, args.reps))
        print(json.dumps(runs[-1]), flush=True)
    model, d, _, vp0 = c4_problem(vb, torch)
    runs.append(run(vb, torch, 'c4_chol', model, vb.MultivariateT(d, 100, seed=1, reparam='cholesky'),
                    vp0.cpu().numpy(), args.n_c4, peak, args.reps))
    print(json.dumps(runs[-1]), flush=True)
    out = {'gpu': gpu_identity(), 'fp64_matmul_peak_tflops': peak,
           'peak_note': 'torch.matmul fp64 4096^3 measured in this run (best of 10, bench.matmul_peak_tflops)',
           'kernel_note': 'CUDA events around vb_mvt_target_log_weights_f64 alone over all n draws (sqrtm map formed '
                          'beforehand; chunked theta_out without the model for c4_chol), best of --reps',
           'end_to_end_note': 'host clock around vi_diagnostics(keep_samples=False) ending in a device synchronise, '
                              'after a warm-up call at n = 2e5: draws, log-weights, PSIS and bounds',
           'runs': runs}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(out, f, indent=1)
    print(json.dumps({'wrote': args.out}))


if __name__ == '__main__':
    main()
