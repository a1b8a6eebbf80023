#!/usr/bin/env python
"""bench.py -- ELBO-gradient iterations/s on BASELINE.json configs[1]:
Bayesian logistic regression N=1e6, d=512, S=256, MFGaussian + RMSProp (synthetic data).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--path f64|fast] [--impl reference] [--dump-outputs DIR]

One "step" = the three hot-path calls of the reference loop (optimization.py:95-98):
objective(var_param) (Philox draws -> sweep over all N observations -> value + gradient),
descent_direction(grad) and update -- here ONE enqueue of three kernels (viabel_b200.engine.FusedStep,
the same object RMSProp.optimize() drives), replayed from a CUDA graph.  For N > 1 the observations
are sharded over the ranks (strong scaling of the same problem) and the S + 2d partial sums are
exchanged inside the step's last kernel through peer memory.  Prints ONE JSON line (rank 0).

`--impl reference` times the CPU arm: the numpy float64 oracle (a port: the reference's own
autograd path cannot run in this image) on the FULL problem, row blocks spread over all host cores.
"""
import os
import sys

if '--impl' in sys.argv and 'reference' in sys.argv:
    # the CPU arm spreads row blocks over a thread pool: one BLAS thread per worker (torchrun exports
    # OMP_NUM_THREADS=1 anyway; set before numpy loads its BLAS)
    for _v in ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'MKL_NUM_THREADS'):
        os.environ[_v] = '1'

import argparse
import json
import subprocess
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_OBS, DIM, S_MC = 1000000, 512, 256
DATA_SEED, DRAW_SEED = 20260117, 1234
CPU_SAMPLE_ROWS = 200000


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--path', default=os.environ.get('VB_BENCH_PATH', 'auto'), choices=['auto', 'f64', 'fast'])
    ap.add_argument('--n-obs', type=int, default=N_OBS)
    ap.add_argument('--dim', type=int, default=DIM)
    ap.add_argument('--mc', type=int, default=S_MC)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-psis', action='store_true')
    ap.add_argument('--no-f64', action='store_true')
    ap.add_argument('--no-graph', action='store_true', help='enqueue every step from Python instead of replaying graphs')
    ap.add_argument('--psis-draws', type=int, default=100000000)
    ap.add_argument('--ref-seconds', type=float, default=None,
                    help='time budget of the reference arm: it stops timing early (after at least 2 steps) when the '
                         'next step would exceed it; without it, all --steps steps are timed')
    ap.add_argument('--config', default='c2', choices=['c2', 'c4'], help='c2: the headline ELBO-gradient bench; c4: BASELINE configs[3]')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed step computed (value, grad, var_param) as DIR/<name>.npy (float64)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'b200' or args.config != 'c2'):
        ap.error('--dump-outputs applies to the headline ELBO-gradient bench (--impl b200 --config c2)')
    return args


def workload_name(N, d, S):
    return 'bayes-logistic N=%d d=%d S=%d MFGaussian+RMSProp (BASELINE configs[%d])' % (
        N, d, S, 2 if (N, d) == (10000000, 1024) else 1)


# ----------------------------------------------------------------------------------------------
# CPU arm: the numpy oracle (a port of the reference iteration; the reference's own autograd
# path cannot run in this image -- autograd/paragami are absent), row blocks over all host cores.
# ----------------------------------------------------------------------------------------------
def host_problem(n_rows, d, seed):
    rs = np.random.RandomState(seed)
    X = rs.standard_normal((n_rows, d))
    beta = rs.standard_normal(d) / np.sqrt(d)
    y = np.where(rs.random_sample(n_rows) < 1.0 / (1.0 + np.exp(-(X @ beta))), 1.0, -1.0)
    return X, y


class CpuIteration(object):
    """The oracle's ELBO step with the N observations split into row blocks evaluated by a thread pool
    (numpy releases the GIL in BLAS and in its elementwise loops): the same arithmetic as
    oracle.viabel_oracle.elbo_step_logistic, using every host core."""

    def __init__(self, X, y, workers):
        from concurrent.futures import ThreadPoolExecutor
        from oracle import viabel_oracle as vo
        self.vo, self.X, self.y = vo, X, y
        self.workers = max(1, int(workers))
        self.pool = ThreadPoolExecutor(self.workers)
        n = X.shape[0]
        nb = max(self.workers * 4, 1)
        edges = np.linspace(0, n, nb + 1).astype(np.int64)
        self.blocks = [(int(a), int(b)) for a, b in zip(edges[:-1], edges[1:]) if b > a]
        self.state = {}

    def model(self, theta):
        vo = self.vo
        lp, gp = vo.gauss_prior(theta, 10.0)

        def part(blk):
            f, G = vo.logistic_logp_grad(theta, self.X[blk[0]:blk[1]], self.y[blk[0]:blk[1]], 10.0, chunk=16384)
            return f - lp, G - gp

        f, G = lp.copy(), gp.copy()
        for fb, Gb in self.pool.map(part, self.blocks):
            f += fb
            G += Gb
        return f, G

    def step(self, vp, eps, lr=0.01):
        vo = self.vo
        value, grad, _ = vo.exclusive_kl_meanfield(vp, eps, self.model)
        return vp - lr * vo.rmsprop_direction(self.state, grad), value, grad


def cpu_iterations(n_rows, d, S, steps, warmup, budget_s=None):
    """(seconds per iteration, iterations timed) of the oracle on n_rows observations."""
    from oracle import viabel_oracle as vo
    X, y = host_problem(n_rows, d, DATA_SEED)
    # one BLAS thread per pool worker (the workers already cover every core; nested BLAS threading oversubscribes the
    # host 16-fold and was measured 6x slower).  The --impl reference arm sets the same through the environment.
    try:
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=1)
    except Exception:
        pass
    it = CpuIteration(X, y, os.cpu_count() or 1)
    rs = np.random.RandomState(DRAW_SEED)
    vp = vo.mfg_init_param(d)
    times = []
    t_start = time.perf_counter()
    for k in range(warmup + steps):
        eps = rs.standard_normal((S, d))
        t0 = time.perf_counter()
        vp, _, _ = it.step(vp, eps)
        dt = time.perf_counter() - t0
        if k >= warmup:
            times.append(dt)
        if budget_s is not None and len(times) >= 2 and time.perf_counter() - t_start + dt > budget_s:
            break
    return float(np.mean(times)), len(times), it.workers


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    sec, done, workers = cpu_iterations(args.n_obs, args.dim, args.mc, args.steps, max(1, min(args.warmup, 1)),
                                        budget_s=args.ref_seconds)
    value = 1.0 / sec
    budget = '' if args.ref_seconds is None else ' (time budget %.0f s)' % args.ref_seconds
    sample = ('oracle (numpy float64 port of the reference iteration) on all %d rows, %d of the %d requested '
              'steps timed%s, row blocks over %d threads' % (args.n_obs, done, args.steps, budget, workers))
    line = {
        'impl': 'reference', 'metric': 'elbo_grad_iters_per_sec', 'value': value, 'unit': 'iter/s',
        'n_gpus': args.gpus, 'steps': done, 'warmup': max(1, min(args.warmup, 1)), 'ms_per_step': sec * 1e3,
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f64',
        'data': 'synthetic', 'extrapolated': False,
        'config': {'workload': workload_name(args.n_obs, args.dim, args.mc)},
        'cpu_baseline': {'value': value, 'unit': 'iter/s', 'cores': workers, 'kind': 'port', 'sample': sample},
        'e2e': {'value': value, 'unit': 'iter/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------
# GPU arm
# ----------------------------------------------------------------------------------------------
class ClockSampler(object):
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile('w+', suffix='.csv', delete=False)
        try:
            self.p = subprocess.Popen(['nvidia-smi', '-i', str(index), '--query-gpu=' + self.Q,
                                       '--format=csv,noheader,nounits', '-lms', '100'],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons, power = [], [], set(), []
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ln in self.f.read().splitlines():
            parts = [x.strip() for x in ln.split(',')]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
                power.append(float(parts[2]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(nm)
        self.f.close()
        os.unlink(self.f.name)
        if sm:
            busy = [s for s, p in zip(sm, power) if p > 0.5 * max(power)] or sm
            out = {'sm_mhz': float(np.median(busy)), 'sm_max_mhz': float(max(mx)), 'reasons': sorted(reasons),
                   'samples': len(sm), 'power_w_max': max(power)}
        return out


def profiled_traffic(*kernels):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the named kernels, from the committed
    ncu --set full captures (profiles/traffic_r02.json, else _r01); None when a kernel has not been captured."""
    for name in ('traffic_r02.json', 'traffic_r01.json'):
        try:
            with open(os.path.join(ROOT, 'profiles', name)) as f:
                t = json.load(f)
            return float(sum(t[k] for k in kernels))
        except (OSError, KeyError, ValueError):
            continue
    return None


def measured_peak(name, fallback):
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            return float(json.load(f)[name]), 'MEASURED_PEAKS.json'
    except Exception:
        return fallback, 'fallback (B200_PROFILING.md)'


def matmul_peak_tflops(torch, dtype, tf32, n, sustained=False):
    """Same method as MEASURED_PEAKS.json's `how`: torch.matmul n^3 (2 n^3 flop) with CUDA events -- best of 10
    (burst), or, with sustained=True, back to back for ~0.7 s and then the mean of 10 more (the figure to hold a
    kernel timed inside a long step against: the boxes of this pool power-cap after a few hundred ms of load)."""
    torch.backends.cuda.matmul.allow_tf32 = tf32
    a = torch.randn(n, n, device='cuda', dtype=dtype)
    b = torch.randn(n, n, device='cuda', dtype=dtype)
    best = 1e9
    for i in range(12):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch.matmul(a, b)
        e1.record()
        torch.cuda.synchronize()
        if i >= 2:
            best = min(best, e0.elapsed_time(e1) * 1e-3)
    if sustained:
        reps = max(10, int(0.7 / best))
        for _ in range(reps):
            torch.matmul(a, b)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            torch.matmul(a, b)
        e1.record()
        torch.cuda.synchronize()
        best = e0.elapsed_time(e1) * 1e-3 / 10
    torch.backends.cuda.matmul.allow_tf32 = False
    return 2.0 * n ** 3 / best / 1e12


def psis_draws(torch, n, dev, seed):
    """log p - log q of a t_10 target under a t_40 proposal, summed over two coordinates (heavy-ish tail)."""
    gen = torch.Generator(device=dev)
    gen.manual_seed(seed)
    lw = torch.zeros(n, device=dev, dtype=torch.float64)
    for _ in range(2):
        z = torch.randn(n, generator=gen, device=dev, dtype=torch.float64)
        lw += -5.5 * torch.log1p(z * z / 10.0) + 20.5 * torch.log1p(z * z / 40.0)
        del z
    return lw


def bench_psis(torch, vb, args):
    """Second headline metric (BASELINE.json: 'PSIS draws/s'): psislw + CUBO/ELBO moments on n
    float64 log-weights resident in HBM (BASELINE configs[4] size, one GPU).  HBM roofline with
    24 algorithmic bytes per draw (lw read twice, smoothed weights written once)."""
    n = args.psis_draws
    lw = psis_draws(torch, n, 'cuda', DATA_SEED + 5)
    out = torch.empty_like(lw)
    # its own steady state: let the GPU leave the power-capped state of the tensor-core legs (1 s idle), then run the
    # PSIS pipeline back to back for ~0.3 s before the timed repetitions
    torch.cuda.synchronize()
    time.sleep(1.0)
    for _ in range(600):
        vb.psislw_device(lw, out)
    torch.cuda.synchronize()
    reps = 20
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        _, res, _, _ = vb.psislw_device(lw, out)
    e1.record()
    torch.cuda.synchronize()
    sec = e0.elapsed_time(e1) * 1e-3 / reps
    r = res.cpu().numpy()
    # diagnostics-only mode (k-hat and the CUBO / ELBO moments, no smoothed output): 16 algorithmic bytes per draw
    for _ in range(2):
        vb.psislw_device(lw, None)
    e0.record()
    for _ in range(reps):
        vb.psislw_device(lw, None)
    e1.record()
    torch.cuda.synchronize()
    sec_diag = e0.elapsed_time(e1) * 1e-3 / reps
    hbm, how = measured_peak('hbm_gbs', 6650.0)
    achieved = 24.0 * n / sec / 1e9
    # end to end from HOST memory through the public API call: H2D of the weights, PSIS, D2H of k-hat and the
    # smoothed weights (pinned buffers; a PCIe-bound number, reported for completeness)
    m2 = min(n, 100000000)            # configs[4]'s own size: 0.8 GB each way
    host = torch.empty(m2, dtype=torch.float64).pin_memory()
    host.copy_(lw[:m2])
    hout = torch.empty_like(host).pin_memory()
    dev_in = torch.empty(m2, device='cuda', dtype=torch.float64)
    for rep in range(2):                  # the second repetition is the timed one (pages touched, workspace cached)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        dev_in.copy_(host, non_blocking=True)
        _, res2, _, _ = vb.psislw_device(dev_in, dev_in)
        hout.copy_(dev_in, non_blocking=True)
        k2 = float(res2[0].item())
        torch.cuda.synchronize()
        e2e = m2 / (time.perf_counter() - t0)
    cpu = None
    if not args.no_cpu_baseline:
        from oracle import viabel_oracle as vo
        m = min(n, 10000000)
        sample = lw[:m].cpu().numpy()
        t0 = time.perf_counter()
        with np.errstate(all='ignore'):
            o, k = vo.psislw_argsort_1d(sample)
            vo.divergence_bound(o)
        cpu = {'value': m / (time.perf_counter() - t0), 'unit': 'draws/s', 'cores': 1, 'kind': 'port',
               'sample': 'numpy oracle with the reference\'s argsort structure (_psis.py:163-203) + divergence_bound '
                         'on the first %d draws' % m}
    del lw, out
    return {'metric': 'psis_draws_per_sec', 'value': n / sec, 'unit': 'draws/s', 'n_draws': n, 'ms': sec * 1e3,
            'khat': float(r[0]), 'n_tail': int(r[2]), 'status': int(r[6]),
            'roofline': {'bound': 'hbm', 'achieved': achieved, 'peak': hbm, 'unit': 'GB/s', 'frac': achieved / hbm,
                         'traffic': profiled_traffic('psis_pass_a_kernel', 'psis_pass_b_kernel') if n == 100000000 else None,
                         'traffic_note': 'the two streaming passes (the short kernels between them touch < 10 MB)',
                         'peak_source': how, 'algorithmic_bytes_per_draw': 24},
            'diagnostics_only': {'value': n / sec_diag, 'unit': 'draws/s', 'ms': sec_diag * 1e3,
                                 'algorithmic_bytes_per_draw': 16, 'achieved_gbs': 16.0 * n / sec_diag / 1e9,
                                 'frac': 16.0 * n / sec_diag / 1e9 / hbm,
                                 'traffic_bytes_per_draw': 8,
                                 'note': 'k-hat + CUBO / ELBO sums in ONE pass over the draws (the sums of the second '
                                         'pass are carried by the first): the kernel moves 8 B/draw, the fraction is '
                                         'quoted on SURVEY 8(d)\'s 16 B/draw definition of the work'},
            'e2e': {'value': e2e, 'unit': 'draws/s', 'n_draws': m2, 'h2d_bytes': m2 * 8,
                    'd2h_bytes': m2 * 8 + 8, 'khat': k2, 'note': 'PCIe-bound'},
            'cpu_baseline': cpu}


def bench_psis_sharded(torch, dist, vb, args, rank, world, dev):
    """BASELINE configs[4]: PSIS of n = 1e8 draws sharded by draw over the ranks (strong scaling of the
    one-GPU leg): pass A + local cutoff per rank, one all-gather of the fixed-size records, replicated
    global select / GPD fit, pass B per rank.  Timed on the device, max over ranks."""
    from viabel_b200.parallel import shard_rows
    n = args.psis_draws
    lo, hi = shard_rows(n, rank, world)
    lw = psis_draws(torch, hi - lo, dev, DATA_SEED + 5 + 1000 * rank)
    out = torch.empty_like(lw)
    sizes = [shard_rows(n, r, world)[1] - shard_rows(n, r, world)[0] for r in range(world)]
    for _ in range(3):
        _, khat, res = vb.psislw_sharded(lw, out=out, sizes=sizes)
    dist.barrier()
    torch.cuda.synchronize()
    reps = 10
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        _, khat, res = vb.psislw_sharded(lw, out=out, sizes=sizes)
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) * 1e-3 / reps], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    sec = float(t.item())
    hbm, how = measured_peak('hbm_gbs', 6650.0)
    achieved = 24.0 * n / sec / 1e9
    # weak scaling beside it: the same pipeline with n draws PER RANK (the replicated select / GPD stages and the
    # exchange are a fixed ~0.3 ms, which a 0.5 ms job cannot hide when split; a world x larger job can)
    del lw, out
    lw = psis_draws(torch, n, dev, DATA_SEED + 5 + 1000 * rank)
    out = torch.empty_like(lw)
    sizes_w = [n] * world
    for _ in range(3):
        vb.psislw_sharded(lw, out=out, sizes=sizes_w)
    dist.barrier()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        _, khat_w, res_w = vb.psislw_sharded(lw, out=out, sizes=sizes_w)
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) * 1e-3 / reps], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    sec_w = float(t.item())
    weak = {'value': n * world / sec_w, 'unit': 'draws/s', 'n_draws': n * world, 'ms': sec_w * 1e3, 'khat': float(khat_w),
            'frac_of_hbm_x_ranks': 24.0 * n * world / sec_w / 1e9 / (hbm * world)}
    del lw, out
    return {'metric': 'psis_draws_per_sec', 'value': n / sec, 'unit': 'draws/s', 'n_draws': n, 'ms': sec * 1e3,
            'weak_scaling': weak,
            'sharding': 'draws over %d ranks (strong scaling of the 1e8-draw column, includes the status read-back)' % world,
            'khat': float(khat), 'n_tail': int(res[2]),
            'roofline': {'bound': 'hbm', 'achieved': achieved, 'peak': hbm * world, 'unit': 'GB/s',
                         'frac': achieved / (hbm * world), 'traffic': None, 'peak_source': how + ' x ranks',
                         'algorithmic_bytes_per_draw': 24}}


def bench_c5(torch, dist, vb, args, rank, world):
    """BASELINE configs[4] END TO END: vi_diagnostics on n = 1e8 draws from a d = 256 Student-t target (df = 10) under
    a mean-field Student-t proposal (df = 40): draw -> log p - log q (fused, streamed: samples[n,d] would be 204.8 GB)
    -> draw-sharded PSIS -> 2-divergence / Wasserstein / error bounds.  ALU bound in the draw stage (2.56e10 Student-t
    variates), so no HBM roofline claim: draws/s and the stage split are reported."""
    import contextlib
    import io
    d, n = 256, args.psis_draws
    rs = np.random.RandomState(20260119)
    loc, scale = rs.randn(d), np.exp(0.25 * rs.randn(d))
    # the proposal is 10 % wider than the target per coordinate: its lighter tails (df 40 vs 10) are then covered and
    # k-hat stays below 0.7, so the whole pipeline (PSIS -> bounds) runs
    vp = np.concatenate([loc + 0.05 * rs.randn(d), np.log(scale) + 0.10 + 0.02 * rs.randn(d)])
    model = vb.StudentTTarget(loc, scale, 10.0)
    approx = vb.MFStudentT(d, 40, seed=DRAW_SEED)
    small = min(n, 2000000)
    with contextlib.redirect_stdout(io.StringIO()):
        vb.vi_diagnostics(vp, model=model, approx=approx, n_samples=small, keep_samples=False)      # warm-up
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rep = vb.vi_diagnostics(vp, model=model, approx=approx, n_samples=n, keep_samples=False)
        torch.cuda.synchronize()
        sec = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([sec], device='cuda', dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        sec = float(t.item())
    return {'metric': 'vi_diagnostics_draws_per_sec', 'value': n / sec, 'unit': 'draws/s', 'n_draws': n, 'dim': d,
            'seconds': sec, 'khat': float(rep['khat']), 'd2': float(rep.get('d2', float('nan'))),
            'W2': float(rep.get('W2', float('nan'))), 'variates_per_sec': n * d / sec,
            'note': 'streamed (no samples[n,d]); draws sharded over %d rank(s); wall clock incl. the host read-backs' % world}


def time_steps(torch, eng, steps, use_graph):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    eng.run(steps, use_graph=use_graph)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3


def device_problem(torch, vb, N, d, S, path, rank=0, world=1, dev='cuda'):
    """(model, approx, objective) of the headline bench on this rank's rows of the seeded N x d problem."""
    from viabel_b200.parallel import shard_rows
    # this rank's rows [lo, hi) of the N x d problem; rank r seeds its rows with DATA_SEED + r
    lo, hi = shard_rows(N, rank, world)
    gen = torch.Generator(device=dev)
    gen.manual_seed(DATA_SEED + 7919)
    beta = torch.randn(d, generator=gen, device=dev, dtype=torch.float64) / np.sqrt(d)
    gen.manual_seed(DATA_SEED + rank)
    X = torch.randn(hi - lo, d, generator=gen, device=dev, dtype=torch.float64)
    p = torch.sigmoid(X @ beta)
    y = torch.where(torch.rand(hi - lo, generator=gen, device=dev, dtype=torch.float64) < p, 1.0, -1.0)
    del p

    model = vb.LogisticRegression(X, y, prior_scale=10.0, sharded=world > 1)
    approx = vb.MFGaussian(d, seed=DRAW_SEED)
    if path == 'fast':
        model.enable_fast_path(approx)    # tcgen05 + TMA, fp16 hi/lo operand splits; fp16-exact draws (see DESIGN 4.2)
    return model, approx, vb.ExclusiveKL(approx, model, S)


def run_b200(args):
    import torch
    import torch.distributed as dist
    import viabel_b200 as vb
    from viabel_b200.engine import FusedStep
    from viabel_b200.parallel import shard_rows

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    dev = torch.device('cuda', local)
    use_graph = not args.no_graph

    N, d, S = args.n_obs, args.dim, args.mc
    lo, hi = shard_rows(N, rank, world)
    path = 'fast' if args.path == 'auto' else args.path
    model, approx, objective = device_problem(torch, vb, N, d, S, path, rank, world, dev)
    opt = vb.RMSProp(0.01)
    eng = FusedStep(objective, opt)       # the object RMSProp.optimize() drives
    eng.set_param(approx.init_param())

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world > 1:
            t = torch.tensor([x], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return x

    eng.run(max(args.warmup, 3), use_graph=use_graph)
    eng.run(16, use_graph=use_graph)      # untimed: both graph shapes (8-step and 1-step) are captured before the clock starts
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    # (1) burst: the first K steps after the warm-up, GPU clocks still at their idle-boost state
    burst = max_over_ranks(time_steps(torch, eng, args.steps, use_graph))
    barrier()
    # the settle phase's length follows the measured rate, so the timed steps restart from the state the burst left
    # (iterate, optimiser state, draw-stream position): they compute the same thing in every run with the same arguments
    start = eng.save_state()
    # (2) settle: the same step for >= 1.2 s, untimed for `value` but reported as `sustained`.  These boxes reach their
    # steady clocks only after a few hundred ms of load (one busy GPU is power-capped DOWN, eight lightly loaded ones
    # clock UP), so a number taken in the first 20 ms describes neither.  Same count on every rank: the step
    # contains the exchange.
    n_sus = max(args.steps, min(20000, int(1.2 / max(burst / args.steps, 1e-5))))
    n_sus = (n_sus + 7) // 8 * 8
    sus = max_over_ranks(time_steps(torch, eng, n_sus, use_graph))
    eng.rewind(start)                     # device-side copies, enqueued behind the settle phase
    # (3) the K timed steps, in the steady state, back to back with the settle phase (no idle gap)
    elapsed = max_over_ranks(time_steps(torch, eng, args.steps, use_graph))
    barrier()
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, t in (('value', eng.value), ('grad', eng.grad), ('var_param', eng.vp)):
            np.save(os.path.join(args.dump_outputs, name + '.npy'), t.cpu().numpy())
    ms_per_step = elapsed / args.steps * 1e3
    clocks = sampler.stop() if sampler else None
    eng.check_comm()
    finite = bool(torch.isfinite(eng.vp).all())

    # ---- end-to-end through the public API with HOST buffers (numpy in, numpy out), as a viabel user calls it:
    #      objective(var_param) -> descent_direction -> update on the host (optimization.py:95-98) -----------
    vp_host = approx.init_param()
    opt2 = vb.RMSProp(0.01)
    # same steady state as `value`: the loop runs for ~0.6 s (same count on every rank) before its K timed steps
    n_pre = max(3, int(0.6 / max(elapsed / args.steps, 1e-5)))
    for _ in range(n_pre):
        v, g = objective(vp_host)
        vp_host = vp_host - 0.01 * opt2.descent_direction(g)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        v, g = objective(vp_host)                   # H2D var_param, D2H value + gradient (pinned, inside one graph)
        vp_host = vp_host - 0.01 * opt2.descent_direction(g)
    barrier()
    e2e_sec = (time.perf_counter() - t0) / args.steps
    if world > 1:
        t = torch.tensor([e2e_sec], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_sec = float(t.item())

    # ---- dominant kernel alone (the sweep through the C ABI), CUDA events on the launching stream, in the same
    #      steady state: back to back for ~0.5 s, then the mean of the next launches --------
    theta = approx.sample(torch.as_tensor(approx.init_param(), device=dev), S)
    base = approx.last_base
    for _ in range(max(3, int(0.5 / max(elapsed / args.steps, 1e-5)))):
        model.sweep(theta, base, None, True)
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = max(10, min(args.steps, 50))
    k0.record()
    for _ in range(reps):
        model.sweep(theta, base, None, True)
    k1.record()
    torch.cuda.synchronize()
    sweep_sec = k0.elapsed_time(k1) * 1e-3 / reps

    psis = c5 = None
    if not args.no_psis:
        del eng
        if world > 1:
            psis = bench_psis_sharded(torch, dist, vb, args, rank, world, dev)
        elif rank == 0:
            psis = bench_psis(torch, vb, args)
        c5 = bench_c5(torch, dist, vb, args, rank, world)

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    flops = 4.0 * (hi - lo) * d * S                  # algorithmic flops of one sweep on this rank
    bf16_peak, how = measured_peak('bf16_tflops', 1590.0)
    bf16_sus, _ = measured_peak('bf16_tflops_sustained', 1390.0)
    if path == 'f64':
        peak = matmul_peak_tflops(torch, torch.float64, False, 4096)
        peak_note = 'cuBLAS fp64 matmul 4096^3 measured in this run (torch.matmul, 2 n^3 flop, best of 10, CUDA events)'
    else:
        peak = matmul_peak_tflops(torch, torch.float32, True, 8192, sustained=True)
        peak_burst = matmul_peak_tflops(torch, torch.float32, True, 8192)
        peak_note = ('cuBLAS tf32 matmul 8192^3 measured in this run with the method of MEASURED_PEAKS.json (torch.matmul, '
                     '2 n^3 flop, CUDA events): SUSTAINED figure (back to back for 0.7 s, then the mean of 10), because the '
                     'kernel is timed inside a long run; burst (best of 10) = %.1f.  SURVEY 8(d) names this denominator' % peak_burst)
    achieved = flops / sweep_sec / 1e12
    traffic = None
    if path == 'fast' and world == 1 and (N, d, S) == (1000000, 512, 256):
        traffic = profiled_traffic('glm_fast_pair_kernel')       # ncu --set full capture of this very launch shape
    roofline = {'bound': 'tensor', 'achieved': achieved, 'peak': peak, 'unit': 'TFLOP/s',
                'frac': achieved / peak, 'traffic': traffic, 'kernel': 'glm_sweep_%s' % path,
                'kernel_ms': sweep_sec * 1e3, 'peak_note': peak_note,
                'bf16_peak_tflops': bf16_peak, 'bf16_peak_source': how,
                'bf16_peak_sustained_tflops': bf16_sus,
                'frac_bf16_algorithmic': achieved / bf16_sus,
                'frac_bf16_executed': ((1.5 if os.environ.get('VB_FAST_FP8', '1') != '0' else 2.0) * achieved / bf16_sus)
                                      if path == 'fast' else None,
                'executed_note': ('GEMM1 = one fp16 pass + two e5m2 correction passes at twice the fp16 rate, GEMM2 = one fp16 '
                                  'pass: 1.5x the algorithmic flops in fp16-pass units (VB_FAST_FP8=0: three fp16 passes, 2x)'),
                'algorithmic_flops_per_launch': flops, 'algorithmic_bytes_per_launch': (hi - lo) * d * 4.0 if path == 'fast'
                else (hi - lo) * d * 8.0}

    # ---- the exact FP64 path of the same config (BASELINE configs[1]: "FP64 and FP32 paths") ----
    f64_leg = None
    if path == 'fast' and world == 1 and not args.no_f64:
        model.path = 'f64'
        approx64 = vb.MFGaussian(d, seed=DRAW_SEED)
        obj64 = vb.ExclusiveKL(approx64, model, S)
        eng64 = FusedStep(obj64, vb.RMSProp(0.01))
        eng64.set_param(approx64.init_param())
        eng64.run(2, use_graph=False)
        torch.cuda.synchronize()
        n64 = 5
        sec64 = time_steps(torch, eng64, n64, False) / n64
        peak64 = matmul_peak_tflops(torch, torch.float64, False, 4096)
        f64_leg = {'value': 1.0 / sec64, 'unit': 'iter/s', 'ms_per_step': sec64 * 1e3, 'steps': n64, 'dtype': 'f64',
                   'roofline': {'bound': 'tensor', 'achieved': flops / sec64 / 1e12, 'peak': peak64, 'unit': 'TFLOP/s',
                                'frac': flops / sec64 / 1e12 / peak64, 'traffic': profiled_traffic('glm_sweep_f64_kernel'),
                                'peak_note': 'cuBLAS fp64 matmul 4096^3 measured in this run (best of 10); whole step timed',
                                'algorithmic_bytes_per_launch': (hi - lo) * d * 8.0}}
        model.path = 'fast'
        del eng64

    cpu_baseline = None
    if not args.no_cpu_baseline and world == 1:
        rows = min(CPU_SAMPLE_ROWS, N)
        sec, done, workers = cpu_iterations(rows, d, S, 3, 1)
        sec *= N / rows
        cpu_baseline = {'value': 1.0 / sec, 'unit': 'iter/s', 'cores': workers, 'kind': 'port',
                        'sample': 'numpy float64 oracle, %d iterations on %d of %d rows over %d threads, time scaled '
                                  'linearly in rows (the --impl reference arm runs all rows)' % (done, rows, N, workers)}

    line = {
        'metric': 'elbo_grad_iters_per_sec', 'value': 1e3 / ms_per_step, 'unit': 'iter/s',
        'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3), 'ms_per_step': ms_per_step,
        'settle_steps': 16 + args.steps + n_sus,
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None,
        'dtype': 'f64' if path == 'f64' else ('f16+e5m2-corrections/f32' if os.environ.get('VB_FAST_FP8', '1') != '0'
                                             else 'f16x2-split/f32'),
        'data': 'synthetic',
        'config': {'workload': workload_name(N, d, S),
                   'path': path, 'rows_per_rank': hi - lo, 'l2': 'inputs larger than L2 (X = %.2f GB per rank)'
                   % ((hi - lo) * d * (4 if path == 'fast' else 8) / 1e9),
                   'step': 'CUDA graph replay of 3 kernels (pre | sweep | post)' if use_graph else '3 kernels enqueued from Python',
                   'exchange': 'in-kernel one-shot all-reduce over peer memory' if world > 1 else 'none',
                   'draws': 'fp16-exact Philox normals (enable_fast_path sets quantize_draws=2)' if path == 'fast' else 'fp64 Philox normals'},
        'timing': 'K steps timed in the steady state: after W warm-up steps, K burst steps and a %d-step settle phase' % n_sus,
        'burst': {'value': args.steps / burst, 'unit': 'iter/s', 'ms_per_step': burst / args.steps * 1e3, 'steps': args.steps,
                  'note': 'the first K steps after the warm-up (the round-1 definition of `value`)'},
        'sustained': {'value': n_sus / sus, 'unit': 'iter/s', 'ms_per_step': sus / n_sus * 1e3, 'steps': n_sus},
        'clocks': clocks,
        'e2e': {'value': 1.0 / e2e_sec, 'unit': 'iter/s', 'h2d_bytes_per_step': 2 * d * 8,
                'd2h_bytes_per_step': (1 + 2 * d) * 8,
                'note': 'objective(var_param) with numpy in / numpy out + the host RMSProp update, K steps after %d settle '
                        'steps; the host gaps between steps lower the GPU duty cycle, so the power-capped clock sits '
                        'slightly higher than in the back-to-back graph replay that `value` times' % n_pre},
        'gpu_launches': (3 if path == 'fast' else 7) * args.steps,
        'finite': finite,
        'roofline': roofline,
        'f64': f64_leg,
        'cpu_baseline': cpu_baseline,
        'psis': psis,
        'c5_vi_diagnostics': c5,
    }
    print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_c4(args):
    """BASELINE configs[3]: hierarchical linear regression with d = 2048 latents (G = 65 groups x p = 31 coefficients +
    31 hyper-means + log tau + log sigma, 200 observations per group; SURVEY 8(d)), full-rank MultivariateT(df = 100),
    AlphaDivergence(alpha = 2), S = 256, RMSProp step.  One iteration = unpack -> Sigma = L L^T -> eigh (cuSOLVER, the
    one library call) -> reparameterise -> grouped model kernel -> cotangent GEMMs -> fused RMSProp.  Roofline: the
    float64 tensor-pipe GEMMs of csrc/gemm_f64.cu (executed flops 8 d^3 + 8 S d^2) against the cuBLAS fp64 matmul peak."""
    import torch
    import viabel_b200 as vb
    torch.cuda.set_device(0)
    G, p, n_per, S = 65, 31, 200, args.mc
    rs = np.random.RandomState(20260118)
    N = G * n_per
    group = np.repeat(np.arange(G), n_per)
    X = rs.randn(N, p)
    m = rs.randn(p)
    beta = m + 0.5 * rs.randn(G, p)
    y = np.sum(X * beta[group], axis=1) + 0.3 * rs.randn(N)
    model = vb.HierarchicalLinearRegression(X, y, group, G)
    d = model.dim
    approx = vb.MultivariateT(d, 100, seed=DRAW_SEED)
    objective = vb.AlphaDivergence(approx, model, S, 2.0)
    # 2.1 M free parameters: RMSProp's first steps move every Cholesky entry by the learning rate, and a unit-lower-
    # triangular factor with +-lr/0.1 below the diagonal stays well conditioned only for small lr
    opt = vb.RMSProp(0.0005)
    # start near a sensible scale (Sigma = 0.01 I): the reference's init Sigma = 10 I overflows the likelihood scale
    vp0 = approx.init_param()
    F = np.zeros((d, d))
    F[np.diag_indices(d)] = 0.5 * np.log(0.01)
    vp0[d:] = F[np.tril_indices(d)]
    vp0[:G * p] = beta.reshape(-1)
    vp0[G * p:G * p + p] = m
    vp = torch.as_tensor(vp0, device='cuda')

    def step():
        value, grad = objective(vp)
        opt._fused_step(vp, grad, False)
        return value

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    sampler = ClockSampler(0)
    steps = args.steps
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        v = step()
    e1.record()
    torch.cuda.synchronize()
    sec = e0.elapsed_time(e1) * 1e-3 / steps
    finite = bool(torch.isfinite(vp).all()) and bool(torch.isfinite(v))

    def timed(fn, reps=3):
        fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            out = fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) * 1e-3 / reps, out

    _, L, hl = approx.unpack(vp)
    t_sigma, Sigma = timed(lambda: approx.sigma(L))
    t_eigh, (w, V) = timed(lambda: approx._eigh(Sigma))
    chi2, z = approx.base_draws(S)
    t_tr, (theta, P, zu2) = timed(lambda: approx.transform(vp, chi2, z, w, V))
    t_model, (f, Gm) = timed(lambda: model.logp_and_grad(theta))
    out = torch.empty(1 + vp.numel(), dtype=torch.float64, device='cuda')
    ws = torch.empty(vb._lib.lib.vb_mvt_objective_workspace_bytes(S, d), dtype=torch.uint8, device='cuda')
    ptr = vb._lib.ptr
    t_obj, _ = timed(lambda: vb._lib.check(vb._lib.lib.vb_mvt_objective_f64(
        ptr(L), ptr(hl), ptr(w), ptr(V), ptr(P), ptr(zu2), ptr(f), ptr(Gm), S, d, 100.0, 2, 2.0, ptr(out[:1]), ptr(out[1:]),
        ptr(ws), ws.numel(), vb._lib.stream())))
    clocks = sampler.stop()
    gemm_flops = 8.0 * d ** 3 + 8.0 * S * d * d
    t_gemm = t_sigma + t_tr + t_obj
    peak = matmul_peak_tflops(torch, torch.float64, False, 4096)
    achieved = gemm_flops / t_gemm / 1e12
    # end to end with host buffers: numpy var_param in, numpy value + gradient out
    vp_host = vp.cpu().numpy()
    for _ in range(2):
        objective(vp_host)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    n_e2e = max(2, min(steps, 5))
    for _ in range(n_e2e):
        vh, gh = objective(vp_host)
        vp_host = vp_host - 0.01 * gh / (np.abs(gh) + 1.0)
    e2e = (time.perf_counter() - t0) / n_e2e
    line = {
        'metric': 'alpha_grad_iters_per_sec', 'value': 1.0 / sec, 'unit': 'iter/s', 'n_gpus': 1, 'steps': steps,
        'warmup': max(args.warmup, 3), 'ms_per_step': sec * 1e3, 'higher_is_better': True, 'scaling': 'strong',
        'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': 'hier-linear d=%d (G=%d p=%d, %d obs) MultivariateT(df=100) AlphaDivergence(alpha=2) S=%d + RMSProp '
                               '(BASELINE configs[3])' % (d, G, p, N, S),
                   'l2': 'parameter and cotangent matrices (7 x d^2 x 8 B = %.0f MB) exceed L2' % (7 * d * d * 8 / 1e6)},
        'clocks': clocks,
        'e2e': {'value': 1.0 / e2e, 'unit': 'iter/s', 'h2d_bytes_per_step': int(vp.numel()) * 8,
                'd2h_bytes_per_step': (1 + int(vp.numel())) * 8},
        'gpu_launches': 24 * steps, 'finite': finite,
        'roofline': {'bound': 'tensor', 'achieved': achieved, 'peak': peak, 'unit': 'TFLOP/s', 'frac': achieved / peak,
                     'traffic': None, 'kernel': 'gemm_f64_kernel (8 launches per iteration)', 'kernel_ms': t_gemm * 1e3,
                     'peak_note': 'cuBLAS fp64 matmul 4096^3 measured in this run (best of 10)',
                     'executed_flops_per_iteration': gemm_flops},
        'stages_ms': {'sigma_gemm': t_sigma * 1e3, 'eigh_cusolver': t_eigh * 1e3, 'transform_gemms': t_tr * 1e3,
                      'model_grouped_kernel': t_model * 1e3, 'objective_gemms': t_obj * 1e3},
        'cpu_baseline': None,
    }
    print(json.dumps(line))


def main():
    args = parse()
    if args.impl == 'reference':
        run_reference(args)
    elif args.config == 'c4':
        run_c4(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
