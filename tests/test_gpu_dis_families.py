"""DISInclusiveKL for MultivariateT (both reparameterisations), LRGaussian and NVPFlow on the device.

Kernels (vb_mvt_score_f64, vb_lr_score_f64) element by element against the long-double references of
tests/_dis_score_ref.py under the bound

    |dev - ref| <= 64 u (d + k + n / 32 + 64) cond mag

where mag is the sum of the absolute summands of each output (the reference returns it) and cond the condition number
of L (MultivariateT, whose inverse the kernel forms) or of Sigma (LRGaussian); then the objective end to end against a
numpy restatement of the reference's DIS steps (objectives.py:283-416) built from the oracle's samplers and log
densities, the golden file of the unmodified reference through LRGaussian(k = 0), convergence, synchronisation and
error paths."""
import math

import numpy as np
import pytest
import torch

import _dis_score_ref as R
import _mf_kernels_ref as MR
from conftest import relerr
from _problems import target_params

pytestmark = pytest.mark.gpu
U = 2.0 ** -53
SENT = 1234.5


@pytest.fixture(scope='module')
def vb():
    import viabel_b200
    return viabel_b200


@pytest.fixture(scope='module')
def vo():
    from oracle import viabel_oracle
    return viabel_oracle


def _dev(a, dtype=torch.float64):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device='cuda')


def _mvt_vp(d, rs, cond=4.0, mu_scale=1.0):
    """L = diag(l) (I + N), l log-spaced over [1, cond], N strictly lower with entries 0.3 / sqrt(d) N(0, 1)"""
    ldiag = np.exp(np.linspace(0.0, math.log(cond), d))
    rs.shuffle(ldiag)
    N = np.tril(rs.randn(d, d), -1) * (0.3 / math.sqrt(d))
    L = ldiag[:, None] * (np.eye(d) + N)
    F = np.tril(L, -1) + np.diag(np.log(np.diag(L)))
    return np.concatenate([mu_scale * rs.randn(d), F[np.tril_indices(d)]]), L


def _call_score(vb, kind, vpd, xd, idx, w, scale, n, d, k=0, df=5.0, P=None):
    """run one score call into NaN-filled outputs followed by sentinels; returns the output vector (host)"""
    lib, ptr, st = vb._lib.lib, vb._lib.ptr, vb._lib.stream()
    nv = vpd.numel()
    out = torch.full((1 + nv + 16,), float('nan'), dtype=torch.float64, device='cuda')
    out[1 + nv:] = SENT
    if kind == 'mvt':
        ws = torch.empty(lib.vb_mvt_score_workspace_bytes(n, d), dtype=torch.uint8, device='cuda')
        vb._lib.check(lib.vb_mvt_score_f64(ptr(vpd), ptr(xd), ptr(idx), ptr(w), scale, n, d, df, ptr(out[:1]),
                                           ptr(out[1:1 + nv]), ptr(ws), ws.numel(), st))
    else:
        ws = torch.empty(lib.vb_lr_score_workspace_bytes(n, d, k), dtype=torch.uint8, device='cuda')
        vb._lib.check(lib.vb_lr_score_f64(ptr(vpd), ptr(P), ptr(xd), ptr(idx), ptr(w), scale, n, d, k, ptr(out[:1]),
                                          ptr(out[1:1 + nv]), ptr(ws), ws.numel(), st))
    h = out.cpu().numpy()
    assert np.all(h[1 + nv:] == SENT), 'write past the gradient'
    assert np.all(np.isfinite(h[:1 + nv]))
    return h[:1 + nv]


def _check(h, ref, n, d, k, cond, tag):
    value, grad, mag, vmag = ref
    tol = 64 * U * (d + k + n / 32 + 64) * cond
    gv = np.asarray(grad, dtype=np.longdouble)
    err = np.abs(h[1:].astype(np.longdouble) - gv)
    bound = tol * np.asarray(mag, dtype=np.longdouble) + 1e-300
    worst = float(np.max(err / bound))
    assert worst <= 1.0, (tag, worst, int(np.argmax(err / bound)))
    assert float(abs(np.longdouble(h[0]) - value)) <= tol * float(vmag), (tag, 'value')


def _rows(rs, n, m, d, shift):
    x = rs.randn(m, d) + shift
    idx = rs.randint(0, m, size=n)                    # unordered, repeated
    return x, idx


MVT_CASES = [(1, 1), (31, 7), (32, 33), (33, 1025), (63, 1), (64, 7), (65, 33), (129, 1025), (257, 33), (257, 1025)]


@pytest.mark.parametrize('d,n', MVT_CASES)
@pytest.mark.parametrize('special', ['plain', 'shift', 'cond'])
def test_mvt_score_elementwise(vb, d, n, special):
    rs = np.random.RandomState(7 * d + n)
    cond = 1e6 if special == 'cond' else 4.0
    vp, L = _mvt_vp(d, rs, cond=cond, mu_scale=1e3 if special == 'shift' else 1.0)
    x, idx = _rows(rs, n, max(3, n // 2), d, vp[:d])
    w = rs.rand(n) + 0.05
    df = 3.5 if d % 2 else 40.0
    vpd, xd, idxd, wd = _dev(vp), _dev(x), _dev(idx, torch.int64), _dev(w)
    h = _call_score(vb, 'mvt', vpd, xd, idxd, wd, 0.3, n, d, df=df)
    ref = R.mvt_score(vp, x, idx, w, 0.3, df, dtype=np.longdouble)
    _check(h, ref, n, d, 0, np.linalg.cond(L), ('mvt', d, n, special))
    # w = NULL equals explicit ones bit for bit; three repeated calls are bitwise equal
    a = _call_score(vb, 'mvt', vpd, xd, idxd, None, 0.3, n, d, df=df)
    b = _call_score(vb, 'mvt', vpd, xd, idxd, _dev(np.ones(n)), 0.3, n, d, df=df)
    c = _call_score(vb, 'mvt', vpd, xd, idxd, None, 0.3, n, d, df=df)
    assert np.array_equal(a, b) and np.array_equal(a, c)
    assert np.array_equal(h, _call_score(vb, 'mvt', vpd, xd, idxd, wd, 0.3, n, d, df=df))


LR_CASES = [(1, 0, 1), (31, 1, 7), (32, 8, 33), (33, 64, 1025), (63, 0, 33), (64, 1, 1025), (65, 8, 1), (129, 64, 7),
            (257, 8, 1025), (257, 64, 33)]


@pytest.mark.parametrize('d,k,n', LR_CASES)
@pytest.mark.parametrize('special', ['plain', 'shift'])
def test_lr_score_elementwise(vb, d, k, n, special):
    from viabel_b200.convenience import _lr_projection
    rs = np.random.RandomState(11 * d + k + n)
    vp = np.concatenate([(1e3 if special == 'shift' else 1.0) * rs.randn(d), 0.3 * rs.randn(d),
                         rs.randn(d * k) / math.sqrt(max(k, 1))])
    x, idx = _rows(rs, n, max(3, n // 2), d, vp[:d])
    w = rs.rand(n) + 0.05
    approx = vb.LRGaussian(d, k=k)
    vpd = _dev(vp)
    P = _lr_projection(vpd, approx)
    xd, idxd, wd = _dev(x), _dev(idx, torch.int64), _dev(w)
    h = _call_score(vb, 'lr', vpd, xd, idxd, wd, 0.7, n, d, k=k, P=P)
    ref = R.lr_score(vp, x, idx, w, 0.7, k, dtype=np.longdouble)
    B = vp[2 * d:].reshape(d, k)
    cond = np.linalg.cond(B @ B.T + np.diag(np.exp(2 * vp[d:2 * d])))
    _check(h, ref, n, d, k, cond, ('lr', d, k, n, special))
    a = _call_score(vb, 'lr', vpd, xd, idxd, None, 0.7, n, d, k=k, P=P)
    b = _call_score(vb, 'lr', vpd, xd, idxd, _dev(np.ones(n)), 0.7, n, d, k=k, P=P)
    c = _call_score(vb, 'lr', vpd, xd, idxd, None, 0.7, n, d, k=k, P=P)
    assert np.array_equal(a, b) and np.array_equal(a, c)


def test_scores_past_65535_row_tiles(vb):
    """d = 1 with more than 65535 tiles of 32 (MultivariateT) or 64 (LRGaussian) rows"""
    from viabel_b200.convenience import _lr_projection
    rs = np.random.RandomState(3)
    n = 64 * 65536 + 7
    x = rs.randn(n, 1)
    vp = np.array([0.2, 0.3])
    h = _call_score(vb, 'mvt', _dev(vp), _dev(x), None, None, 1.0 / n, n, 1, df=6.0)
    _check(h, R.mvt_score(vp, x, None, None, 1.0 / n, 6.0, dtype=np.longdouble), n, 1, 0, 1.0, 'mvt big n')
    vp = np.array([0.2, 0.1, 0.8])
    vpd = _dev(vp)
    P = _lr_projection(vpd, vb.LRGaussian(1, k=1))
    h = _call_score(vb, 'lr', vpd, _dev(x), None, None, 1.0 / n, n, 1, k=1, P=P)
    _check(h, R.lr_score(vp, x, None, None, 1.0 / n, 1, dtype=np.longdouble), n, 1, 1, 2.0, 'lr big n')


@pytest.mark.parametrize('reparam', ['sqrtm', 'cholesky'])
def test_mvt_score_full_size(vb, reparam):
    """d = 2048, n = 1024 through the objective's own score call, against the float64 reference at 1e-10"""
    d, n = 2048, 1024
    rs = np.random.RandomState(2048)
    vp, _ = _mvt_vp(d, rs)
    x, idx = _rows(rs, n, 700, d, vp[:d])
    approx = vb.MultivariateT(d, 8.0, reparam=reparam)
    obj = vb.DISInclusiveKL(approx, vb.Model(lambda z: -0.5 * (z ** 2).sum(dim=1)), n, 100, vb.MFGaussian(d),
                            np.zeros(2 * d))
    value, grad = obj._score(_dev(vp), _dev(x), _dev(idx, torch.int64), None, 0.01)
    v0, g0, _, _ = R.mvt_score(vp, x, idx, None, 0.01, 8.0)
    assert relerr(float(value[0]), v0) < 1e-10
    assert relerr(grad.cpu().numpy(), g0) < 1e-10


def test_lr_score_d2048(vb):
    from viabel_b200.convenience import _lr_projection
    d, k, n = 2048, 64, 1025
    rs = np.random.RandomState(5)
    vp = np.concatenate([rs.randn(d), 0.3 * rs.randn(d), rs.randn(d * k) / 8])
    x, idx = _rows(rs, n, 600, d, vp[:d])
    vpd = _dev(vp)
    h = _call_score(vb, 'lr', vpd, _dev(x), _dev(idx, torch.int64), None, 0.5, n, d, k=k,
                    P=_lr_projection(vpd, vb.LRGaussian(d, k=k)))
    v0, g0, _, _ = R.lr_score(vp, x, idx, None, 0.5, k)
    assert relerr(h[0], v0) < 1e-10 and relerr(h[1:], g0) < 1e-10


# ---- objective: pinned to the reference, end to end, convergence ----------------------------------------------------
@pytest.mark.parametrize('mode', ['nores1', 'res1', 'res3'])
def test_lr_k0_reproduces_mfg_golden(vb, golden, mode):
    """LRGaussian(4, k=0) is MFGaussian draw for draw: the reference's mfg DIS calls, value, gradient and epsilon"""
    g = golden('dis_objective')
    mean, sd = target_params(4, seed=14)
    resample, batches = mode.startswith('res'), int(mode[-1])
    obj = vb.DISInclusiveKL(vb.LRGaussian(4, k=0), vb.GaussianTarget(mean, sd), 60, 20, vb.MFGaussian(4),
                            np.concatenate([np.zeros(4), np.ones(4)]), use_resampling=resample,
                            num_resampling_batches=batches)
    tag = 'dis_obj/mfg/%s' % mode
    np.random.seed(846)
    for c in range(4):
        key = '%s/call%d' % (tag, c)
        base = (np.empty((60, 0)), g[key + '/base']) if key + '/base' in g else None
        v, gr = obj(g[key + '/var_param'], base=base)
        eps_ref = float(g[key + '/eps'])
        assert obj._eps == eps_ref if eps_ref in (0.0, 1.0) else abs(obj._eps - eps_ref) < 1e-12, key
        assert relerr(v, g[key + '/value']) < 1e-10, key
        assert relerr(gr, g[key + '/grad']) < 1e-10, key


def _restated_dis(calls, sampler, logq, logp, lprior, score, S, ess_target, batch, resample, batches):
    """the reference's DIS steps (objectives.py:317-416) in numpy: one (value, grad, eps) per call"""
    out, eps, state = [], 1.0, None
    for c, (vp, base) in enumerate(calls):
        if not resample or c % batches == 0:
            x = sampler(vp, base)
            lq, lp, lpr = logq(vp, x), logp(x), lprior(x)
            res = MR.dis_bisection(lpr, lp, lq, eps, 1.0, ess_target, 50)
            eps, mid = res['eps'], res['mid']
            w = np.exp(mid * lpr + (1 - mid) * lp - lq)
            state = (x, w)
        x, w = state
        if not resample:
            v, g = score(vp, x, None, w, 1.0 / S)
        else:
            p = w / w.sum()
            try:
                idx = np.random.choice(S, size=batch, p=p)
            except ValueError:
                idx = np.random.choice(S, size=batch, p=p / p.sum())
            v, g = score(vp, x, idx, None, float(w.sum()) / S / batch)
        out.append((v, g, eps))
    return out


def _gauss_target(vb, d, seed):
    mean, sd = target_params(d, seed=seed)
    return vb.GaussianTarget(mean, sd), (lambda x: np.sum(-0.5 * ((x - mean) / sd) ** 2 - np.log(sd)
                                                          - 0.5 * math.log(2 * math.pi), axis=1))


def _run_e2e(vb, vo, approx, d, vp0, base_fn, sampler, logq, score, resample, batches, fd_grad=False):
    S, ess_target = 60, 20
    target, logp = _gauss_target(vb, d, 21)
    prior_vp = np.concatenate([np.zeros(d), np.full(d, 0.5)])
    obj = vb.DISInclusiveKL(approx, target, S, ess_target, vb.MFGaussian(d), prior_vp, use_resampling=resample,
                            num_resampling_batches=batches)
    rs = np.random.RandomState(99)
    np.random.seed(846)
    calls, got, vp = [], [], vp0
    for c in range(4):
        base = base_fn(rs, S) if (not resample or c % batches == 0) else None
        v, g = obj(vp, base=base)
        calls.append((vp, base))
        got.append((v, g, obj._eps))
        vp = vp - 0.02 * g
    np.random.seed(846)
    want = _restated_dis(calls, sampler, logq, logp, lambda x: vo.mfg_log_density(prior_vp, x), score, S, ess_target,
                         obj._resampling_batch_size, resample, batches)
    for c, ((v, g, e), (v0, g0, e0)) in enumerate(zip(got, want)):
        assert e == e0 if e0 in (0.0, 1.0) else abs(e - e0) < 1e-12, c
        assert relerr(v, v0) < 1e-10, c
        assert relerr(g, g0) < (1e-5 if fd_grad else 1e-10), (c, relerr(g, g0))


@pytest.mark.parametrize('reparam', ['sqrtm', 'cholesky'])
@pytest.mark.parametrize('resample,batches', [(False, 1), (True, 1), (True, 3)])
def test_mvt_dis_end_to_end(vb, vo, reparam, resample, batches):
    d, df = 4, 7.0
    mean, sd = target_params(d, seed=21)
    vp0 = vo.mvt_pack(mean + 0.3, np.diag(sd ** 2) * 1.5 + 0.1)

    def sampler(vp, base):
        chi2, z = base
        if reparam == 'sqrtm':
            return vo.mvt_sample(vp, chi2, z, df)
        mu, L = vo.mvt_unpack(vp, d)
        return mu + (z @ L.T) / np.sqrt(chi2 / df)[:, None]
    _run_e2e(vb, vo, vb.MultivariateT(d, df, reparam=reparam), d, vp0,
             lambda rs, S: (rs.chisquare(df, S), rs.randn(S, d)), sampler,
             lambda vp, x: vo.mvt_log_density(vp, x, df),
             lambda vp, x, idx, w, sc: R.mvt_score(vp, x, idx, w, sc, df)[:2], resample, batches)


@pytest.mark.parametrize('k', [1, 8])
@pytest.mark.parametrize('resample,batches', [(False, 1), (True, 3)])
def test_lr_dis_end_to_end(vb, vo, k, resample, batches):
    d = 9
    mean, sd = target_params(d, seed=21)
    rs = np.random.RandomState(k)
    vp0 = np.concatenate([mean + 0.3, np.log(sd), 0.3 * rs.randn(d * k)])
    _run_e2e(vb, vo, vb.LRGaussian(d, k=k), d, vp0, lambda rs, S: (rs.randn(S, k), rs.randn(S, d)),
             lambda vp, base: vo.lr_sample(vp, base[0], base[1]), lambda vp, x: vo.lr_log_density(vp, x, k),
             lambda vp, x, idx, w, sc: R.lr_score(vp, x, idx, w, sc, k)[:2], resample, batches)


@pytest.mark.parametrize('resample,batches', [(False, 1), (True, 3)])
def test_nvpflow_dis_end_to_end(vb, vo, resample, batches):
    """value against the oracle's flow log density at 1e-10; gradient against central differences of it"""
    d, hidden, pairs = 3, 6, 2
    layers = [[d, hidden], [hidden, d]]
    masks = np.array([[0, 1, 1], [1, 0, 0]] * pairs)
    prior_param = np.concatenate([np.zeros(d), np.zeros(d)])
    fam = vb.NVPFlow(layers, layers, masks, vb.MFGaussian(d), prior_param, d)
    shapes = [tuple(s) for s in layers]
    vp0 = 0.1 * np.random.RandomState(4).randn(fam.var_param_dim)

    def logq(vp, x):
        return vo.nvp_log_density(vp, shapes, shapes, masks, x, prior_param)

    def score(vp, x, idx, w, sc):
        xs = x if idx is None else x[idx]
        c = sc * (np.ones(xs.shape[0]) if w is None else w)
        f = lambda v: -np.sum(c * logq(v, xs))
        h, g = 1e-6, np.zeros(vp.size)
        for i in range(vp.size):
            e = np.zeros(vp.size)
            e[i] = h
            g[i] = (f(vp + e) - f(vp - e)) / (2 * h)
        return f(vp), g
    _run_e2e(vb, vo, fam, d, vp0, lambda rs, S: rs.randn(S, d),
             lambda vp, base: vo.nvp_g(vp, shapes, shapes, masks, vo.mfg_sample(prior_param, base)), logq, score,
             resample, batches, fd_grad=True)


def _gaussian_model(vb, m, P):
    Pt, mt = torch.as_tensor(P, device='cuda'), torch.as_tensor(m, device='cuda')
    return vb.Model(lambda theta: -0.5 * (((theta - mt) @ Pt) * (theta - mt)).sum(dim=1))


@pytest.mark.parametrize('family', ['mvt-sqrtm', 'mvt-cholesky', 'lr'])
def test_dis_adam_converges(vb, family):
    """DIS + Adam recovers a correlated 3-D Gaussian (rank-1 plus diagonal covariance) to 0.2 in mean and covariance"""
    m = np.array([1.0, -2.0, 0.5])
    b = np.array([0.8, -0.6, 0.4])
    C = np.outer(b, b) + np.diag([0.5, 0.8, 0.3])
    np.random.seed(0)
    if family == 'lr':
        approx = vb.LRGaussian(3, seed=2, k=1)
    else:
        approx = vb.MultivariateT(3, 100, seed=2, reparam=family.split('-')[1])
    obj = vb.DISInclusiveKL(approx, _gaussian_model(vb, m, np.linalg.inv(C)), 400, 100, vb.MFGaussian(3),
                            np.concatenate([np.zeros(3), np.log(3.0) * np.ones(3)]), num_resampling_batches=4)
    opt = vb.Adam(0.02)
    opt.progress = False
    res = opt.optimize(3000, obj, approx.init_param())
    mean, cov = approx.mean_and_cov(res['opt_param'])
    assert np.max(np.abs(mean - m)) < 0.2, mean
    assert np.max(np.abs(cov - C)) < 0.2, cov


# ---- synchronisation and errors -------------------------------------------------------------------------------------
def test_cholesky_score_enqueues_no_sync(vb):
    d, n = 70, 50
    rs = np.random.RandomState(8)
    vp, _ = _mvt_vp(d, rs)
    x, idx = _rows(rs, n, 40, d, vp[:d])
    obj = vb.DISInclusiveKL(vb.MultivariateT(d, 5.0, reparam='cholesky'), vb.Model(lambda z: -(z ** 2).sum(dim=1)), n,
                            10, vb.MFGaussian(d), np.zeros(2 * d))
    vpd, xd, idxd, wd = _dev(vp), _dev(x), _dev(idx, torch.int64), _dev(rs.rand(n))
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode('error')
    try:
        v, g = obj._score(vpd, xd, idxd, wd, 0.5)
        v2, g2 = obj._score(vpd, xd, None, None, 0.5)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert bool(torch.isfinite(g).all()) and bool(torch.isfinite(g2).all())


def test_score_cabi_errors(vb):
    lib, ptr, st, cl = vb._lib.lib, vb._lib.ptr, vb._lib.stream(), vb._lib
    d, n, k = 5, 6, 2
    rs = np.random.RandomState(0)
    vp, _ = _mvt_vp(d, rs)
    vpd, xd = _dev(vp), _dev(rs.randn(n, d))
    out = torch.full((1 + vp.size,), 3.5, dtype=torch.float64, device='cuda')
    need = lib.vb_mvt_score_workspace_bytes(n, d)
    assert need > 0 and lib.vb_mvt_score_workspace_bytes(0, d) == 0
    ws = torch.full((need,), 7, dtype=torch.uint8, device='cuda')

    def mvt(vp_=vpd, x_=xd, n_=n, d_=d, df=5.0, val=out[:1], nbytes=need, ws_=ws):
        return lib.vb_mvt_score_f64(ptr(vp_), ptr(x_), None, None, 1.0, n_, d_, df, ptr(val), ptr(out[1:]), ptr(ws_), nbytes, st)
    assert mvt(vp_=None) == cl.VB_ERR_INVALID_ARG
    assert mvt(x_=None) == cl.VB_ERR_INVALID_ARG
    assert mvt(val=None) == cl.VB_ERR_INVALID_ARG
    assert mvt(n_=0) == cl.VB_ERR_INVALID_ARG
    assert mvt(d_=0) == cl.VB_ERR_INVALID_ARG
    assert mvt(df=2.0) == cl.VB_ERR_INVALID_ARG
    assert mvt(nbytes=need - 1) == cl.VB_ERR_WORKSPACE
    assert mvt(ws_=None) == cl.VB_ERR_WORKSPACE
    assert mvt(n_=2 ** 31, nbytes=2 ** 62) == cl.VB_ERR_UNSUPPORTED

    vpl = _dev(rs.randn(2 * d + d * k))
    P = _dev(rs.randn(k, k + d))
    outl = torch.full((1 + 2 * d + d * k,), 3.5, dtype=torch.float64, device='cuda')
    needl = lib.vb_lr_score_workspace_bytes(n, d, k)
    assert needl > 0 and lib.vb_lr_score_workspace_bytes(n, d, -1) == 0
    wsl = torch.full((needl,), 7, dtype=torch.uint8, device='cuda')

    def lr(vp_=vpl, P_=P, x_=xd, n_=n, d_=d, k_=k, val=outl[:1], nbytes=needl):
        return lib.vb_lr_score_f64(ptr(vp_), ptr(P_), ptr(x_), None, None, 1.0, n_, d_, k_, ptr(val), ptr(outl[1:]),
                                   ptr(wsl), nbytes, st)
    assert lr(vp_=None) == cl.VB_ERR_INVALID_ARG
    assert lr(P_=None) == cl.VB_ERR_INVALID_ARG
    assert lr(x_=None) == cl.VB_ERR_INVALID_ARG
    assert lr(val=None) == cl.VB_ERR_INVALID_ARG
    assert lr(n_=-1) == cl.VB_ERR_INVALID_ARG
    assert lr(d_=0) == cl.VB_ERR_INVALID_ARG
    assert lr(k_=-1) == cl.VB_ERR_INVALID_ARG
    assert lr(nbytes=needl - 1) == cl.VB_ERR_WORKSPACE
    assert lr(n_=2 ** 31, nbytes=2 ** 62) == cl.VB_ERR_UNSUPPORTED
    torch.cuda.synchronize()
    assert bool((out == 3.5).all()) and bool((ws == 7).all())
    assert bool((outl == 3.5).all()) and bool((wsl == 7).all())


def test_objective_errors(vb):
    d = 3
    tgt = vb.Model(lambda z: -0.5 * (z ** 2).sum(dim=1))
    approx = vb.MultivariateT(d, 5.0)                                  # sqrtm mode
    obj = vb.DISInclusiveKL(approx, tgt, 20, 5, vb.MFGaussian(d), np.zeros(2 * d))
    F = np.diag([0.0, 0.0, -13.0])                                     # an eigenvalue of Sigma = e^-26 < 1e-10
    with pytest.raises(NotImplementedError):
        obj(np.concatenate([np.zeros(d), F[np.tril_indices(d)]]))
    with pytest.raises(ValueError):
        obj(np.zeros(approx.var_param_dim + 1))
    lr = vb.DISInclusiveKL(vb.LRGaussian(d, k=1), tgt, 20, 5, vb.MFGaussian(d), np.zeros(2 * d))
    with pytest.raises(ValueError):
        lr(np.zeros(2 * d + d + 1))
    nn = vb.NeuralNet([[d, 4], [4, d]])
    with pytest.raises(NotImplementedError):
        vb.DISInclusiveKL(nn, tgt, 20, 5, vb.MFGaussian(d), np.zeros(2 * d))(np.zeros(nn.var_param_dim))
