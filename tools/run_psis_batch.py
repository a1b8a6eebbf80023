"""Batched PSIS (vb_psislw_batch_f64) timed on one GPU in one process.

    python tools/run_psis_batch.py [--reps 3] [--out profiles/psis_batch.json]

1. The card's name, power limit and maximum SM clock (nvidia-smi), and the device-to-device copy bandwidth of a 4 GB
   buffer measured in this run (read + write bytes over CUDA-event time): the denominator of every share below.
2. Kernel time (CUDA events, after one warm-up call, median of --reps) of psisloo's form (out = NULL, loo: 8 bytes
   per entry) and of 2-D psislw with an output (16 bytes per entry) at (n, m) = (1000, 1e6), (4000, 1e6) and
   (max_n, 1e5) with Reff = 1, and psisloo's form at (4000, 1e6) with Reff = 0.1.  Every input is larger than L2.
   Columns are normal log-weights with a per-column scale in [0.5, 2.5], so the fit and the smoothing run.
3. (max_n + 1, 2000): the one-column route 2-D psislw takes above the limit (every column enqueued, one read of the
   result rows), host clock around the call.
4. The loop 2-D psislw ran before the batched kernel existed (the one-column pipeline and a blocking read of its
   result per column) on 1000 columns of n = 4000, alternated with one batched launch on the same columns.
5. End to end from numpy at (4000, 1e5): psislw and psisloo, host clock, including the host-device copies.
Prints one JSON line and writes it to --out.  Needs a CUDA device.
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


def event_time(torch, fn, reps):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b) * 1e-3)
    return float(np.median(ts)), ts


def copy_bandwidth(torch, reps):
    src = torch.empty(2 ** 29, dtype=torch.float64, device='cuda').fill_(1.0)      # 4 GB
    dst = torch.empty_like(src)
    t, _ = event_time(torch, lambda: dst.copy_(src), reps + 2)
    bw = 2 * src.numel() * 8 / t
    del src, dst
    torch.cuda.empty_cache()
    return bw


def columns(torch, n, m, seed):
    """[m, n] contiguous (column j of the n x m matrix is row j): normal log-weights, per-column scale"""
    g = torch.Generator(device='cuda').manual_seed(seed)
    x = torch.empty((m, n), dtype=torch.float64, device='cuda')
    x.normal_(generator=g)
    x.mul_(torch.empty((m, 1), dtype=torch.float64, device='cuda').uniform_(0.5, 2.5, generator=g))
    return x


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'psis_batch.json'))
    args = ap.parse_args()
    import torch
    import viabel_b200 as vb
    from viabel_b200 import _psis
    torch.cuda.set_device(0)
    rep = dict(gpu=gpu_info())
    bw = copy_bandwidth(torch, args.reps)
    rep['copy_bandwidth_GBps'] = bw / 1e9
    max_n = _psis.psis_batch_max_n(1.0)
    rep['max_n'] = {str(r): _psis.psis_batch_max_n(r) for r in (1.0, 0.3, 0.1, 0.05)}

    kern = []
    for n, m, reff in ((1000, 10 ** 6, 1.0), (4000, 10 ** 6, 1.0), (max_n, 10 ** 5, 1.0), (4000, 10 ** 6, 0.1)):
        cols = columns(torch, n, m, 7 + n)
        lw = cols.t()
        modes = [('psisloo', 8)] if reff != 1.0 else [('psisloo', 8), ('psislw_out', 16)]
        for mode, bpe in modes:
            out = torch.empty_like(cols).t() if mode == 'psislw_out' else None
            t, ts = event_time(torch, lambda: _psis.psislw_batch_device(lw, out, reff, want_loo=mode == 'psisloo'),
                               args.reps)
            rate = bpe * n * m / t
            kern.append(dict(mode=mode, n=n, m=m, reff=reff, seconds=t, all_seconds=ts, bytes_per_entry=bpe,
                             GBps=rate / 1e9, share_of_copy_bw=rate / bw, us_per_column_per_sm=t / m * 148e6,
                             columns_per_s=m / t))
            del out
        del cols, lw
        torch.cuda.empty_cache()
    rep['kernel'] = kern

    # above the limit: the one-column pipeline, every column enqueued, one read of the result rows
    n, m = max_n + 1, 2000
    cols = columns(torch, n, m, 11)
    _psis._psis_columns(cols[:4].clone(), 1.0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    _psis._psis_columns(cols, 1.0)
    t = time.perf_counter() - t0
    rep['per_column_route'] = dict(n=n, m=m, seconds=t, us_per_column=t / m * 1e6, GBps=16 * n * m / t / 1e9)
    del cols
    torch.cuda.empty_cache()

    # the parent's 2-D loop (one pipeline run and one blocking result read per column) against one batched launch
    n, m = 4000, 1000
    base = columns(torch, n, m, 13)
    old_t, new_t = [], []

    def old_loop():
        c = base.clone()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(m):
            _psis._psis_column(c[i], c[i], 1.0, False)
        return time.perf_counter() - t0

    def new_call():
        c = base.clone()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        _, k, _, _ = _psis.psislw_batch_device(c.t(), c.t(), 1.0)
        k.cpu()
        return time.perf_counter() - t0
    old_loop(), new_call()
    for _ in range(args.reps):
        old_t.append(old_loop())
        new_t.append(new_call())
    rep['vs_per_column_loop'] = dict(n=n, m=m, loop_seconds=old_t, batched_seconds=new_t,
                                     loop_us_per_column=float(np.median(old_t)) / m * 1e6,
                                     batched_us_per_column=float(np.median(new_t)) / m * 1e6,
                                     speedup=float(np.median(old_t) / np.median(new_t)))
    del base

    # end to end from numpy
    n, m = 4000, 10 ** 5
    rs = np.random.RandomState(17)
    X = rs.standard_normal((n, m)) * rs.uniform(0.5, 2.5, size=m)
    vb.psislw(X[:, :8])
    vb.psisloo(X[:, :8])
    t0 = time.perf_counter()
    vb.psislw(X)
    t_lw = time.perf_counter() - t0
    t0 = time.perf_counter()
    vb.psisloo(X)
    t_loo = time.perf_counter() - t0
    rep['end_to_end_numpy'] = dict(n=n, m=m, psislw_seconds=t_lw, psisloo_seconds=t_loo)

    line = json.dumps(rep)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        f.write(json.dumps(rep, indent=1) + '\n')


if __name__ == '__main__':
    main()
