"""GPU: the fused AlphaDivergence step (engine.cu VB_OBJ_ALPHA, engine.FusedStep).  Oracle parity over three
optimiser steps with injected draws (eager, then graph replay) on both sweeps; the per-step seeded draws; the same
results and the same global numpy RNG state as the per-iteration loop it replaces in RMSProp / Adam / FASO; graph
replay against eager enqueue; the in-kernel exchange with two ranks in one process; the rejections."""
import ctypes

import numpy as np
import pytest
import torch

import _alpha_step_ref as A
from conftest import relerr
from _problems import logistic_problem, target_params

pytestmark = pytest.mark.gpu
TOL64 = 1e-10
TOL_FAST = 1e-4


@pytest.fixture(scope='module')
def vb():
    import viabel_b200
    return viabel_b200


@pytest.fixture(scope='module')
def vo():
    from oracle import viabel_oracle
    return viabel_oracle


class _LocalComm(object):
    """One rank of a communicator whose peers live in this process (vb_comm_connect_ptrs)."""

    def __init__(self, lib, rank, world, slot_bytes):
        self.handle = ctypes.c_void_p()
        hbuf = (ctypes.c_ubyte * 64)()
        assert lib.vb_comm_create(ctypes.byref(self.handle), rank, world, slot_bytes, hbuf) == 0

    @staticmethod
    def connect(lib, comms):
        ptrs = (ctypes.c_void_p * len(comms))(*[lib.vb_comm_buffer(c.handle) for c in comms])
        for c in comms:
            assert lib.vb_comm_connect_ptrs(c.handle, ptrs) == 0


def _family(vb, fam, d, seed=1):
    return vb.MFGaussian(d, seed=seed) if fam == 'gaussian' else vb.MFStudentT(d, 7.5, seed=seed)


def _bases(rs, fam, S, d, n=3):
    return [rs.randn(S, d) if fam == 'gaussian' else rs.standard_t(7.5, size=(S, d)) for _ in range(n)]


def _run_injected(eng, bases):
    """one step per base, eager first and graph-replayed afterwards; (value, grad, param) after each"""
    out = []
    for k, base in enumerate(bases):
        eng.base.copy_(torch.as_tensor(base, device='cuda'))
        eng.run(1, use_graph=(k > 0))
        out.append((float(eng.value[0]), eng.grad.cpu().numpy(), eng.vp.cpu().numpy()))
    return out


@pytest.mark.parametrize('N,d,S', [(1003, 13, 1), (1003, 13, 7), (700, 77, 100), (2048, 300, 256), (600, 20, 2000)])
@pytest.mark.parametrize('fam', ['gaussian', 'student'])
@pytest.mark.parametrize('alpha', [0.5, 2.0, 5.0])
def test_alpha_step_f64_vs_oracle(vb, vo, N, d, S, fam, alpha):
    """float64 sweeps: value, gradient, updated parameter and the value / param / grad histories, RMSProp and Adam"""
    from viabel_b200.engine import FusedStep
    X, y, beta = logistic_problem(N, d, seed=N + d)
    rs = np.random.RandomState(S)
    model = vb.LogisticRegression(X, y, prior_scale=10.0)
    df = None if fam == 'gaussian' else 7.5
    obj = vb.AlphaDivergence(_family(vb, fam, d), model, S, alpha)
    oracle_model = lambda th: vo.logistic_logp_grad(th, X, y, 10.0)
    for opt_name, opt in (('rmsprop', vb.RMSProp(0.01)), ('adam', vb.Adam(0.01))):
        bases = _bases(rs, fam, S, d)
        vp0 = np.concatenate([0.5 * beta, -1.0 + 0.1 * rs.randn(d)])
        ref = A.alpha_loop(vo, vp0, bases, oracle_model, alpha, opt_name, fam, df)
        eng = FusedStep(obj, opt, ring=4, hist_len=3, inject_base=True, want_grad_hist=True)
        assert eng.launches_per_step == 11
        eng.set_param(vp0)
        got = _run_injected(eng, bases)
        for k in range(3):
            assert relerr(got[k][0], ref[k][0]) < TOL64, (opt_name, k, 'value')
            assert relerr(got[k][1], ref[k][1]) < TOL64, (opt_name, k, 'grad')
            assert relerr(got[k][2], ref[k][2]) < TOL64, (opt_name, k, 'param')
        assert relerr(eng.value_hist.cpu().numpy(), [r[0] for r in ref]) < TOL64
        assert relerr(eng.last_rows(eng.param_hist, 3).cpu().numpy(), np.stack([r[2] for r in ref])) < TOL64
        assert relerr(eng.last_rows(eng.grad_hist, 3).cpu().numpy(), np.stack([r[1] for r in ref])) < TOL64


def test_alpha_step_f64_underflowing_weights(vb, vo):
    """log-weights spread over thousands: most weights are exactly zero (tests/test_alpha_step_host.py builds the same
    problem), and the step still matches the oracle"""
    from viabel_b200.engine import FusedStep
    N, d, S, alpha = 2000, 40, 64, 5.0
    X, y, beta = logistic_problem(N, d, seed=9)
    rs = np.random.RandomState(10)
    bases = [rs.randn(S, d) for _ in range(3)]
    vp0 = np.concatenate([beta, 1.5 * np.ones(d)])
    oracle_model = lambda th: vo.logistic_logp_grad(th, X, y, 10.0)
    _, _, lw0 = vo.alpha_divergence_meanfield(vp0, bases[0], oracle_model, alpha)
    assert np.mean(np.exp(lw0 - lw0.max()) ** alpha == 0.0) > 0.5
    model = vb.LogisticRegression(X, y, prior_scale=10.0)
    eng = FusedStep(vb.AlphaDivergence(vb.MFGaussian(d), model, S, alpha), vb.RMSProp(0.01), ring=3, hist_len=3,
                    inject_base=True)
    eng.set_param(vp0)
    got = _run_injected(eng, bases)
    ref = A.alpha_loop(vo, vp0, bases, oracle_model, alpha, 'rmsprop')
    for k in range(3):
        assert relerr(got[k][0], ref[k][0]) < TOL64 and relerr(got[k][1], ref[k][1]) < TOL64
        assert relerr(got[k][2], ref[k][2]) < TOL64


@pytest.mark.parametrize('N,d,S', [(1003, 13, 7), (20000, 512, 256), (4100, 130, 100), (257, 1024, 256)])
@pytest.mark.parametrize('alpha', [0.5, 2.0, 5.0])
def test_alpha_step_fast_vs_oracle(vb, vo, N, d, S, alpha):
    """tensor-core sweeps on fp16-exact injected draws.  Budget (tests/test_gpu_fast.py, DESIGN.md 4.2): 1e-4 plus
    alpha times the weight-averaged log-weight error of the fp32 sweep, measured at the same point through the
    unfused fast path, which runs the same sweep kernel on the same operands."""
    from viabel_b200.engine import FusedStep
    X, y, beta = logistic_problem(N, d, seed=N + d)
    rs = np.random.RandomState(S)
    model = vb.LogisticRegression(X, y, prior_scale=10.0).enable_fast_path()
    oracle_model = lambda th: vo.logistic_logp_grad(th, X, y, 10.0)
    bases = [rs.randn(S, d).astype(np.float16).astype(np.float64) for _ in range(3)]
    vp0 = np.concatenate([beta + 0.01 * rs.randn(d), -3.5 + 0.1 * rs.randn(d)])
    for opt_name, opt in (('rmsprop', vb.RMSProp(0.01)), ('adam', vb.Adam(0.01))):
        approx = vb.MFGaussian(d)
        obj = vb.AlphaDivergence(approx, model, S, alpha)
        eng = FusedStep(obj, opt, ring=4, hist_len=3, inject_base=True, want_grad_hist=True)
        assert eng.launches_per_step == 5
        eng.set_param(vp0)
        state = {}
        steps = []
        for k, base in enumerate(bases):
            vp = eng.vp.cpu().numpy()
            v0, g0, lw0 = vo.alpha_divergence_meanfield(vp, base, oracle_model, alpha)
            obj(vp, base=base)                              # unfused fast path: its fp32 log-weight error
            e = approx.last_log_weights.cpu().numpy() - lw0
            wn = np.exp(alpha * (lw0 - lw0.max()))
            wn /= wn.sum()
            eff = float(np.sum(wn * np.abs(e - e[np.argmax(lw0)])))
            tol = TOL_FAST + 2.0 * alpha * eff
            eng.base.copy_(torch.as_tensor(base, device='cuda'))
            eng.run(1, use_graph=(k > 0))
            v, g = float(eng.value[0]), eng.grad.cpu().numpy()
            assert relerr(v, v0) < TOL_FAST, (opt_name, k, 'value')
            assert relerr(g, g0) < tol, (opt_name, k, 'grad', eff)
            # the update is the oracle's optimiser applied to the step's own gradient (RMSProp's first direction is
            # about sign(g), so an error in a near-zero gradient component moves that component by up to 2 lr)
            dd = vo.rmsprop_direction(state, g) if opt_name == 'rmsprop' else vo.adam_direction(state, g)
            assert relerr(eng.vp.cpu().numpy(), vp - 0.01 * dd) < TOL64, (opt_name, k, 'param')
            steps.append((v, g, eng.vp.cpu().numpy()))
        assert np.array_equal(eng.value_hist.cpu().numpy(), [s[0] for s in steps])
        assert np.array_equal(eng.last_rows(eng.param_hist, 3).cpu().numpy(), np.stack([s[2] for s in steps]))
        assert np.array_equal(eng.last_rows(eng.grad_hist, 3).cpu().numpy(), np.stack([s[1] for s in steps]))


@pytest.mark.parametrize('fam', ['gaussian', 'student'])
@pytest.mark.parametrize('quantize', [0, 2])
def test_alpha_step_draws_are_the_seeded_streams(vb, fam, quantize):
    """the base draws of step t are approx.base_draws(S, seeds[t]) bit for bit, eager and graph-replayed, across a
    wrap of the seed ring; the family's own stream is left alone"""
    from viabel_b200.engine import FusedStep
    N, d, S = 3000, 70, 33                                  # odd S * d
    X, y, beta = logistic_problem(N, d, seed=5)
    model = vb.LogisticRegression(X, y)
    approx, twin = _family(vb, fam, d, seed=77), _family(vb, fam, d, seed=77)
    approx.quantize_draws = twin.quantize_draws = quantize
    eng = FusedStep(vb.AlphaDivergence(approx, model, S, 2.0), vb.RMSProp(0.01), hist_len=5)
    eng.set_param(np.concatenate([beta, -2.0 * np.ones(d)]))
    seeds = np.random.RandomState(3).randint(2 ** 32, dtype=np.uint64, size=8)
    eng.set_seeds(0, seeds[:5])
    for t in range(8):
        if t == 5:
            eng.set_seeds(5, seeds[5:])                     # slots 0..2 again
        eng.run(1, use_graph=(t % 2 == 1))
        assert torch.equal(eng.base, twin.base_draws(S, int(seeds[t]))), t
    assert approx._offset == 0


def _optimize_pair(vb, monkeypatch, run):
    """run(fused) after np.random.seed, fused first, then with the fused path patched off"""
    import viabel_b200.engine as engine
    out, states = {}, {}
    for fused in (True, False):
        if not fused:
            monkeypatch.setattr(engine, 'fused_step_supported', lambda *a, **k: False)
        np.random.seed(2024)
        out[fused] = run()
        states[fused] = np.random.get_state()
    monkeypatch.undo()
    s0, s1 = states[True], states[False]
    assert s0[0] == s1[0] and np.array_equal(s0[1], s1[1]) and tuple(s0[2:]) == tuple(s1[2:])
    return out[True], out[False]


@pytest.mark.parametrize('opt_name', ['rmsprop', 'adam'])
def test_alpha_optimize_matches_unfused_loop(vb, monkeypatch, capsys, opt_name):
    """RMSProp / Adam .optimize on AlphaDivergence: fused == per-iteration loop, 250 iterations in chunks of 100
    (progress bar on), same RNG state afterwards"""
    N, d, S = 4000, 24, 16
    X, y, beta = logistic_problem(N, d, seed=12)
    model = vb.LogisticRegression(X, y)

    def run():
        approx = vb.MFGaussian(d, seed=5)
        opt = vb.RMSProp(0.02) if opt_name == 'rmsprop' else vb.Adam(0.02)
        opt.progress = True
        return opt.optimize(250, vb.AlphaDivergence(approx, model, S, 2.0), np.concatenate([0.5 * beta, -1.5 * np.ones(d)]))

    a, b = _optimize_pair(vb, monkeypatch, run)
    assert relerr(a['value_history'], b['value_history']) < 1e-9
    assert relerr(a['variational_param_history'], b['variational_param_history']) < 1e-9
    assert relerr(a['opt_param'], b['opt_param']) < 1e-9


def test_alpha_faso_matches_unfused_loop(vb, monkeypatch, capsys):
    """FASO on AlphaDivergence(alpha = 2), started from an ELBO fit (where the reference's estimator is stable) and
    stopping at its first MCSE check: fused == per-iteration loop, the same decisions and the same RNG state"""
    N, d, S = 3000, 2, 100
    X, y, beta = logistic_problem(N, d, seed=44)
    model = vb.LogisticRegression(X, y)
    fit = vb.RMSProp(0.05)
    fit.progress = False
    approx = vb.MFGaussian(d, seed=3)
    init = fit.optimize(600, vb.ExclusiveKL(approx, model, 12), approx.init_param())['opt_param']

    def run():
        approx = vb.MFGaussian(d, seed=17)
        sgo = vb.RMSProp(0.01)
        sgo.progress = False
        faso = vb.FASO(sgo, W_min=100, k_check=100, mcse_threshold=1e3, ESS_min=1)
        return faso.optimize(2000, vb.AlphaDivergence(approx, model, S, 2.0), init)

    a, b = _optimize_pair(vb, monkeypatch, run)
    assert a['k_stopped'] is not None and len(a['value_history']) < 2000
    assert a['k_stopped'] == b['k_stopped'] and a['k_conv'] == b['k_conv'] and a['k_Rhat'] == b['k_Rhat']
    assert len(a['value_history']) == len(b['value_history'])
    assert relerr(a['value_history'], b['value_history']) < 1e-9
    assert relerr(a['variational_param_history'], b['variational_param_history']) < 1e-9
    assert relerr(a['grad_history'], b['grad_history']) < 1e-8
    assert relerr(a['opt_param'], b['opt_param']) < 1e-9


@pytest.mark.parametrize('fam', ['gaussian', 'student'])
@pytest.mark.parametrize('quantize', [0, 2])
def test_alpha_optimize_draws_across_chunks(vb, capsys, fam, quantize):
    """RMSProp.optimize with the progress bar on runs chunks of 100 steps, drawing each chunk's seeds before it: the
    last step's draws are base_draws(S, seed) of the seed the per-iteration loop would have drawn for it, at the end of
    the first chunk (100), the first step of the second (101) and inside the third (250)"""
    N, d, S = 3000, 70, 33
    X, y, beta = logistic_problem(N, d, seed=5)
    model = vb.LogisticRegression(X, y)
    twin = _family(vb, fam, d, seed=77)
    twin.quantize_draws = quantize
    for n in (100, 101, 250):
        approx = _family(vb, fam, d, seed=77)
        approx.quantize_draws = quantize
        opt = vb.RMSProp(0.01)
        opt.progress = True
        np.random.seed(n)
        opt.optimize(n, vb.AlphaDivergence(approx, model, S, 2.0), np.concatenate([beta, -2.0 * np.ones(d)]))
        np.random.seed(n)
        seeds = [np.random.randint(2 ** 32, dtype=np.uint64) for _ in range(n)]
        assert torch.equal(approx.last_base, twin.base_draws(S, int(seeds[-1]))), n
        assert approx._offset == 0


def test_alpha_graph_replay_is_bitwise_eager(vb):
    from viabel_b200.engine import FusedStep
    N, d, S = 9000, 128, 64
    X, y, beta = logistic_problem(N, d, seed=3)
    seeds = np.random.RandomState(4).randint(2 ** 32, dtype=np.uint64, size=21)
    for fast in (True, False):
        model = vb.LogisticRegression(X, y)
        if fast:
            model.enable_fast_path()
        outs = []
        for use_graph in (False, True):
            approx = vb.MFGaussian(d, seed=9)
            approx.quantize_draws = 2
            eng = FusedStep(vb.AlphaDivergence(approx, model, S, 2.0), vb.Adam(0.02), ring=8, hist_len=21)
            eng.set_param(approx.init_param())
            eng.set_seeds(0, seeds)
            eng.run(21, use_graph=use_graph)
            outs.append((eng.vp.clone(), eng.value_hist.clone()))
        assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1]), fast


def test_alpha_step_two_ranks_one_process(vb):
    """observations split over two ranks (two engines on two streams, peer buffers connected by pointer), 5 steps with
    two collectives each: the single-rank result, bit-identical parameters and gradients on both ranks"""
    from viabel_b200.engine import FusedStep
    lib = vb._lib.lib
    N, d, S = 1500, 40, 24
    X, y, beta = logistic_problem(N, d, seed=21)
    cut = 700
    rs = np.random.RandomState(2)
    bases = [rs.randn(S, d) for _ in range(5)]
    vp0 = np.concatenate([0.3 * beta, -1.5 * np.ones(d)])
    for fast in (False, True):
        def model_of(Xp, yp):
            m = vb.LogisticRegression(Xp, yp)
            return m.enable_fast_path() if fast else m
        tol = TOL_FAST if fast else TOL64
        single = FusedStep(vb.AlphaDivergence(vb.MFGaussian(d), model_of(X, y), S, 2.0), vb.RMSProp(0.01),
                           inject_base=True)
        single.set_param(vp0)
        comms = [_LocalComm(lib, r, 2, (S + 2 * d) * 8) for r in range(2)]
        _LocalComm.connect(lib, comms)
        engs, streams = [], [torch.cuda.Stream(), torch.cuda.Stream()]
        for r, (lo, hi) in enumerate(((0, cut), (cut, N))):
            eng = FusedStep(vb.AlphaDivergence(vb.MFGaussian(d), model_of(X[lo:hi], y[lo:hi]), S, 2.0),
                            vb.RMSProp(0.01), inject_base=True)
            eng.comm = comms[r]
            eng.set_param(vp0)
            engs.append(eng)
        for k, base in enumerate(bases):
            b = torch.as_tensor(base, device='cuda')
            if fast:
                b = b.to(torch.float16).to(torch.float64)
            for eng in engs + [single]:
                eng.base.copy_(b)
            single.enqueue()
            torch.cuda.synchronize()
            for eng, st in zip(engs, streams):
                with torch.cuda.stream(st):
                    eng.enqueue()
            torch.cuda.synchronize()
            for c in comms:
                assert lib.vb_comm_error(c.handle) == 0
            assert torch.equal(engs[0].vp, engs[1].vp) and torch.equal(engs[0].grad, engs[1].grad), (fast, k)
            assert float(engs[0].value[0]) == float(engs[1].value[0])
            assert relerr(float(engs[0].value[0]), float(single.value[0])) < tol, (fast, k)
            assert relerr(engs[0].grad.cpu().numpy(), single.grad.cpu().numpy()) < tol, (fast, k)
            assert relerr(engs[0].vp.cpu().numpy(), single.vp.cpu().numpy()) < tol, (fast, k)
        del engs
        for c in comms:
            lib.vb_comm_destroy(c.handle)


def test_alpha_step_rejections(vb):
    """bad alpha and missing seeds: VB_ERR_INVALID_ARG; a workspace below vb_mf_step_workspace_bytes: VB_ERR_WORKSPACE"""
    from viabel_b200.engine import FusedStep
    lib = vb._lib.lib
    N, d, S = 500, 10, 8
    X, y, beta = logistic_problem(N, d, seed=1)
    model = vb.LogisticRegression(X, y)
    eng = FusedStep(vb.AlphaDivergence(vb.MFGaussian(d), model, S, 2.0), vb.RMSProp(0.01), hist_len=4)
    eng.set_param(np.zeros(2 * d))
    st = torch.cuda.current_stream().cuda_stream

    def call(ws_bytes=None):
        return lib.vb_mf_step_glm(ctypes.byref(eng.cfg), ctypes.byref(eng.buf), ctypes.byref(eng.mdl), None,
                                  eng.ws.data_ptr(), eng.ws.numel() if ws_bytes is None else ws_bytes, st)

    for bad in (0.0, float('nan'), float('inf'), -float('inf')):
        eng.cfg.alpha = bad
        assert call() == -1, bad
    eng.cfg.alpha = 2.0
    seeds, n = eng.buf.seeds, eng.buf.seed_len
    eng.buf.seeds = None
    assert call() == -1
    eng.buf.seeds, eng.buf.seed_len = seeds, 0
    assert call() == -1
    eng.buf.seed_len = n
    eng.cfg.inject_base = 1
    eng.buf.seeds = None                                    # injected draws need no seeds
    assert call() == 0
    eng.buf.seeds, eng.cfg.inject_base = seeds, 0
    need = lib.vb_mf_step_workspace_bytes(S, d)
    assert need <= eng.ws.numel()
    assert call(1024) == -4
    assert call() == 0
    torch.cuda.synchronize()
    with pytest.raises(ValueError):
        eng.cfg.alpha = float('nan')
        eng.enqueue()


def test_alpha_fused_step_supported_and_fallbacks(vb, capsys):
    """fused_step_supported is False for non-GLM models, non-mean-field families, other optimisers and an alpha the
    kernel rejects; those keep running through the unfused loop"""
    from viabel_b200.engine import fused_step_supported
    N, d, S = 800, 6, 8
    X, y, beta = logistic_problem(N, d, seed=2)
    glm = vb.LogisticRegression(X, y)
    mean, sd = target_params(d, seed=3)
    target = vb.GaussianTarget(mean, sd)
    ok = vb.AlphaDivergence(vb.MFGaussian(d), glm, S, 2.0)
    assert fused_step_supported(ok, vb.RMSProp(0.01)) and fused_step_supported(ok, vb.Adam(0.01))
    assert fused_step_supported(ok) and fused_step_supported(vb.AlphaDivergence(vb.MFStudentT(d, 5.0), glm, S, 0.5))
    cases = [(vb.AlphaDivergence(vb.MFGaussian(d), target, S, 2.0), vb.RMSProp(0.01)),
             (vb.AlphaDivergence(vb.MultivariateT(d, 50.0), glm, S, 2.0), vb.RMSProp(0.001)),
             (ok, vb.Adagrad(0.01)),
             (ok, vb.WindowedAdagrad(0.01))]
    for a in (0.0, float('nan'), float('inf')):
        cases.append((vb.AlphaDivergence(vb.MFGaussian(d), glm, S, a), vb.RMSProp(0.01)))
    for i, (obj, opt) in enumerate(cases):
        assert not fused_step_supported(obj, opt), i
    for i, (obj, opt) in enumerate(cases[:4]):
        opt.progress = False
        res = opt.optimize(3, obj, obj.approx.init_param())
        assert len(res['value_history']) == 3
        if i != 1:
            assert np.all(np.isfinite(res['value_history'])), i
