"""A/B of the fast kernels: parity of gmu / ge / ll against the float64 sweep on small cases, then C2 timing."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import viabel_b200 as vb

def rel(a, b):
    return float((a - b).norm() / b.norm())

def case(N, d, S, reps=3):
    g = torch.Generator(device='cuda'); g.manual_seed(N + d + S)
    X = torch.randn(N, d, generator=g, device='cuda', dtype=torch.float64)
    y = torch.where(torch.rand(N, generator=g, device='cuda', dtype=torch.float64) < 0.5, 1.0, -1.0)
    th = torch.randn(S, d, generator=g, device='cuda', dtype=torch.float64) * 0.05
    bs = torch.randn(S, d, generator=g, device='cuda', dtype=torch.float64).to(torch.float16).to(torch.float64)
    m = vb.LogisticRegression(X, y)
    ref = torch.cat(m.sweep(th, bs, None, True))
    m.enable_fast_path()
    for r in range(reps):
        out = torch.cat(m.sweep(th, bs, None, True))
        torch.cuda.synchronize()
        print('N=%d d=%d S=%d rep %d: ll %.2e gmu %.2e ge %.2e' % (N, d, S, r, rel(out[:S], ref[:S]), rel(out[S:S + d], ref[S:S + d]),
                                                             rel(out[S + d:], ref[S + d:])), flush=True)

if len(sys.argv) > 1 and sys.argv[1] == 'time':
    N, d, S = 1000000, 512, 256
    g = torch.Generator(device='cuda'); g.manual_seed(1)
    X = torch.randn(N, d, generator=g, device='cuda', dtype=torch.float64)
    y = torch.where(torch.rand(N, generator=g, device='cuda', dtype=torch.float64) < 0.5, 1.0, -1.0)
    m = vb.LogisticRegression(X, y).enable_fast_path()
    del X
    th = torch.randn(S, d, generator=g, device='cuda', dtype=torch.float64) * 0.05
    bs = torch.randn(S, d, generator=g, device='cuda', dtype=torch.float64)
    for tot in (False, True):
        for _ in range(3):
            m.sweep(th, bs, None, True, ll_total_only=tot)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20):
            m.sweep(th, bs, None, True, ll_total_only=tot)
        e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 20
        print('C2 sweep ll_total_only=%d %.4f ms  %.1f TFLOP/s algorithmic' % (tot, ms, 4.0 * N * d * S / ms / 1e9))
else:
    for c in [(128, 128, 64), (128, 128, 64), (1003, 13, 7), (300, 256, 256), (257, 1024, 256), (5, 2048, 3), (40000, 64, 256), (100000, 512, 256)]:
        case(*c)
