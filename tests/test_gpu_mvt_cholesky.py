"""GPU: MultivariateT(..., reparam='cholesky') -- theta = mu + L z / u through the triangular float64 tensor-core
kernels of csrc/mvt_chol.cu -- against the numpy reference of tests/_mvt_cholesky_ref.py (1e-10 relative,
norm-wise), tied to the reference-pinned log density and base draws, and checked as an estimator: distribution of the draws, unbiasedness of the gradient,
determinism, no host synchronisation, convergence."""
import math

import numpy as np
import pytest
import torch
from scipy import stats

import _mvt_cholesky_ref as cr
from conftest import relerr
from _problems import hier_problem

pytestmark = pytest.mark.gpu

TOL64 = 1e-10


@pytest.fixture(scope='module')
def vb():
    import viabel_b200
    return viabel_b200


@pytest.fixture(scope='module')
def vo():
    from oracle import viabel_oracle
    return viabel_oracle


def _hier_oracle(vo, hp, chunk=32):
    def om(theta):
        parts = [vo.hier_linear_logp_grad(theta[i:i + chunk], hp['X'], hp['y'], hp['group'], hp['G'], hp['p'])
                 for i in range(0, theta.shape[0], chunk)]
        return np.concatenate([a for a, _ in parts]), np.concatenate([b for _, b in parts])
    return om


def _correlated_point(vo, d, rs, diag=0.9, scale=0.3):
    B = scale * rs.randn(d, d) / np.sqrt(d)
    return vo.mvt_pack(0.2 * rs.randn(d), diag * np.eye(d) + B @ B.T)


@pytest.mark.parametrize('G,p,n_per,S', [(1, 5, 40, 9), (3, 20, 30, 24), (7, 31, 40, 40)])
def test_cholesky_hier_vs_oracle(vb, vo, G, p, n_per, S):
    """Hierarchical linear regression at d = 12, 82, 250: sample, ExclusiveKL and AlphaDivergence(2) value and gradient
    against the numpy Cholesky-mode reference."""
    hp = hier_problem(G=G, p=p, n_per=n_per, seed=31 + G)
    model = vb.HierarchicalLinearRegression(hp['X'], hp['y'], hp['group'], G)
    d = model.dim
    om = _hier_oracle(vo, hp)
    rs = np.random.RandomState(d)
    approx = vb.MultivariateT(d, 100, reparam='cholesky')
    vp = _correlated_point(vo, d, rs)
    chi2, z = rs.chisquare(100, S), rs.randn(S, d)
    x = approx.sample(vp, S, base=(chi2, z))
    assert relerr(x, cr.mvt_sample_cholesky(vp, chi2, z, 100.0)) < TOL64
    v, gr = vb.ExclusiveKL(approx, model, S)(vp, base=(chi2, z))
    v0, g0, _ = cr.exclusive_kl_mvt_cholesky(vp, chi2, z, om, 100.0)
    assert relerr(v, v0) < TOL64 and relerr(gr, g0) < TOL64
    v, gr = vb.AlphaDivergence(approx, model, S, 2.0)(vp, base=(chi2, z))
    v0, g0, _ = cr.alpha_divergence_mvt_cholesky(vp, chi2, z, om, 100.0, 2.0)
    assert relerr(v, v0) < TOL64 and relerr(gr, g0) < TOL64


def test_cholesky_c4_full_size_vs_oracle(vb, vo):
    """BASELINE configs[3] at full size (d = 2048, S = 256, 2 100 224 free parameters) at one correlated point."""
    hp = hier_problem(G=65, p=31, n_per=200, seed=20260118)
    model = vb.HierarchicalLinearRegression(hp['X'], hp['y'], hp['group'], 65)
    d, S = model.dim, 256
    assert d == 2048
    approx = vb.MultivariateT(d, 100, reparam='cholesky')
    assert approx.var_param_dim == 2100224
    rs = np.random.RandomState(4)
    F = np.tril(0.002 * rs.randn(d, d), -1) + np.diag(0.5 * np.log(0.01) + 0.05 * rs.randn(d))
    vp = np.concatenate([0.1 * rs.randn(d), F[np.tril_indices(d)]])
    vp[d - 2:d] = [-1.0, -1.2]                               # log tau, log sigma near the data's scales
    chi2, z = rs.chisquare(100, S), rs.randn(S, d)
    om = _hier_oracle(vo, hp)
    v, gr = vb.ExclusiveKL(approx, model, S)(vp, base=(chi2, z))
    v0, g0, _ = cr.exclusive_kl_mvt_cholesky(vp, chi2, z, om, 100.0)
    assert relerr(v, v0) < TOL64 and relerr(gr, g0) < TOL64
    v, gr = vb.AlphaDivergence(approx, model, S, 2.0)(vp, base=(chi2, z))
    v0, g0, _ = cr.alpha_divergence_mvt_cholesky(vp, chi2, z, om, 100.0, 2.0)
    assert relerr(v, v0) < TOL64 and relerr(gr, g0) < TOL64


@pytest.mark.parametrize('d', [1, 5, 63, 64, 65, 130, 257])
@pytest.mark.parametrize('S', [1, 7, 64, 100])
def test_cholesky_kernels_ragged(vb, vo, d, S):
    """Both kernels through the C ABI at ragged shapes (partial tiles, odd column-block pairs, one sample) against
    numpy, for ExclusiveKL and AlphaDivergence weights, with arbitrary f and G."""
    rs = np.random.RandomState(1000 * d + S)
    df = 5.0
    F = np.tril(rs.randn(d, d), -1) + np.diag(0.3 * rs.randn(d))
    vp = np.concatenate([rs.randn(d), F[np.tril_indices(d)]])
    chi2, z = rs.chisquare(df, S), rs.randn(S, d)
    f, G = rs.randn(S), rs.randn(S, d)
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a), device='cuda')
    vpd, zd, cd, fd, Gd = t(vp), t(z), t(chi2), t(f), t(G)
    lib, ptr, st = vb._lib.lib, vb._lib.ptr, vb._lib.stream()
    theta = torch.empty(S, d, dtype=torch.float64, device='cuda')
    inv_u = torch.empty(S, dtype=torch.float64, device='cuda')
    zu2 = torch.empty(S, dtype=torch.float64, device='cuda')
    vb._lib.check(lib.vb_mvt_chol_transform_f64(ptr(vpd), ptr(zd), ptr(cd), df, S, d, ptr(theta), ptr(inv_u), ptr(zu2), st))
    zu = z / np.sqrt(chi2 / df)[:, None]
    assert relerr(theta.cpu().numpy(), cr.mvt_sample_cholesky(vp, chi2, z, df)) < TOL64
    assert relerr(inv_u.cpu().numpy(), 1.0 / np.sqrt(chi2 / df)) < 1e-14
    assert relerr(zu2.cpu().numpy(), np.sum(zu * zu, axis=1)) < 1e-13
    ws = torch.empty(lib.vb_mvt_chol_objective_workspace_bytes(S, d), dtype=torch.uint8, device='cuda')
    fixed = lambda th: (f, G)
    for objective, alpha in ((vb._lib.OBJ_EXCLUSIVE_KL, 0.0), (vb._lib.OBJ_ALPHA, 1.5)):
        out = torch.full((1 + vp.size,), float('nan'), dtype=torch.float64, device='cuda')
        vb._lib.check(lib.vb_mvt_chol_objective_f64(ptr(vpd), ptr(zd), ptr(inv_u), ptr(zu2), ptr(fd), ptr(Gd), S, d, df, objective,
                                                    alpha, ptr(out[:1]), ptr(out[1:]), ptr(ws), ws.numel(), st))
        if objective == vb._lib.OBJ_ALPHA:
            v0, g0, _ = cr.alpha_divergence_mvt_cholesky(vp, chi2, z, fixed, df, alpha)
        else:
            v0, g0, _ = cr.exclusive_kl_mvt_cholesky(vp, chi2, z, fixed, df)
        o = out.cpu().numpy()
        assert np.isfinite(o).all()                           # every packed entry written
        assert relerr(o[0], v0) < TOL64 and relerr(o[1:], g0) < TOL64


def test_cholesky_log_density_and_base_draws(vb, vo):
    """The eigh-based log_density (pinned to the reference by tests/golden/families.npz) at Cholesky-mode draws equals
    the closed form c - sum F_ii - (df + d)/2 log1p(|z/u|^2 / df); both modes draw the same base variates."""
    d, df, n = 12, 7.0, 300
    rs = np.random.RandomState(12)
    vp = _correlated_point(vo, d, rs)
    a_chol = vb.MultivariateT(d, df, seed=5, reparam='cholesky')
    a_sqrt = vb.MultivariateT(d, df, seed=5)
    x = a_chol.sample(vp, n)
    a_sqrt.sample(vp, n)
    chi2, z = (t.cpu().numpy() for t in a_chol.last_base)
    for t0, t1 in zip(a_chol.last_base, a_sqrt.last_base):
        assert torch.equal(t0, t1)
    zu = z / np.sqrt(chi2 / df)[:, None]
    _, L = vo.mvt_unpack(vp, d)
    closed = (math.lgamma(0.5 * (df + d)) - math.lgamma(0.5 * df) - 0.5 * d * math.log(math.pi * df)
              - np.sum(np.log(np.diag(L))) - 0.5 * (df + d) * np.log1p(np.sum(zu * zu, axis=1) / df))
    assert relerr(a_chol.log_density(vp, x), closed) < TOL64
    # the objectives draw the same way too: chi-square first, then z, from the family's own stream
    model = vb.GaussianTarget(np.zeros(d), np.ones(d))
    vb.ExclusiveKL(a_chol, model, 9)(vp)
    vb.ExclusiveKL(a_sqrt, model, 9)(vp)
    for t0, t1 in zip(a_chol.last_base, a_sqrt.last_base):
        assert torch.equal(t0, t1)


def test_cholesky_distribution(vb, vo):
    """10^6 draws at d = 12: per-coordinate means and per-entry covariances against mean_and_cov, one-sample t-tests
    with p > 1e-4 (the reference tests' criterion)."""
    d, df, n = 12, 100, 10 ** 6
    rs = np.random.RandomState(77)
    vp = _correlated_point(vo, d, rs, diag=0.5, scale=1.0)
    approx = vb.MultivariateT(d, df, seed=11, reparam='cholesky')
    x = approx.sample(vp, n)
    mean, cov = approx.mean_and_cov(vp)
    for j in range(d):
        assert stats.ttest_1samp(x[:, j], mean[j]).pvalue > 1e-4, j
    c = x - mean
    for i in range(d):
        for j in range(i + 1):
            assert stats.ttest_1samp(c[:, i] * c[:, j], cov[i, j]).pvalue > 1e-4, (i, j)


def _gaussian_model(vb, m, P):
    Pt, mt = torch.as_tensor(P, device='cuda'), torch.as_tensor(m, device='cuda')

    def logp(theta):
        r = theta - mt
        return -0.5 * ((r @ Pt) * r).sum(dim=1)
    return vb.Model(logp, lambda theta: -(theta - mt) @ Pt)


@pytest.mark.parametrize('reparam', ['sqrtm', 'cholesky'])
def test_exclusive_kl_gradient_unbiased(vb, vo, reparam):
    """Correlated Gaussian target log p = -(theta - m)^T P (theta - m) / 2: E[grad] is closed form, grad_mu =
    P (mu - m), grad_L = tril(k P L) with k = df / (df - 2), times L_ii on the diagonal, minus 1 there (entropy).
    The mean of 400 independent gradients lies within 5 Monte Carlo standard errors of it, in each mode."""
    d, df, S, n = 4, 8.0, 16, 400
    rs = np.random.RandomState(3)
    B = rs.randn(d, d) / np.sqrt(d)
    P = np.eye(d) + B @ B.T
    m = rs.randn(d)
    vp = _correlated_point(vo, d, rs, diag=0.6, scale=0.8)
    mu, L = vo.mvt_unpack(vp, d)
    k = df / (df - 2.0)
    Fbar = np.tril(k * P @ L)
    Fbar[np.diag_indices(d)] = Fbar[np.diag_indices(d)] * np.diag(L) - 1.0
    g_true = np.concatenate([P @ (mu - m), Fbar[np.tril_indices(d)]])
    approx = vb.MultivariateT(d, df, seed=21, reparam=reparam)
    obj = vb.ExclusiveKL(approx, _gaussian_model(vb, m, P), S)
    vpd = torch.as_tensor(vp, device='cuda')
    grads = torch.stack([obj(vpd)[1] for _ in range(n)]).cpu().numpy()
    se = grads.std(axis=0, ddof=1) / np.sqrt(n)
    assert (se > 0).all()
    assert np.max(np.abs(grads.mean(axis=0) - g_true) / se) < 5.0


def test_cholesky_deterministic_and_no_host_sync(vb, vo):
    """Repeated evaluations on the same inputs give identical bits, and an evaluation plus an RMSProp step with a device
    var_param enqueues no host synchronisation (the eager optimiser loop runs ahead of the GPU)."""
    hp = hier_problem(G=7, p=31, n_per=40, seed=38)
    model = vb.HierarchicalLinearRegression(hp['X'], hp['y'], hp['group'], 7)
    d, S = model.dim, 100
    rs = np.random.RandomState(9)
    vp = torch.as_tensor(_correlated_point(vo, d, rs), device='cuda')
    approx = vb.MultivariateT(d, 100, reparam='cholesky')
    base = approx.base_draws(S)
    for obj in (vb.ExclusiveKL(approx, model, S), vb.AlphaDivergence(approx, model, S, 2.0)):
        v1, g1 = obj(vp, base=base)
        v2, g2 = obj(vp, base=base)
        assert torch.equal(v1, v2) and torch.equal(g1, g2)
        assert bool(torch.isfinite(g1).all())
    opt = vb.RMSProp(1e-3)
    objs = (vb.ExclusiveKL(approx, model, S), vb.AlphaDivergence(approx, model, S, 2.0))
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode('error')
    try:
        for obj in objs:
            for _ in range(2):
                _, g = obj(vp)
                opt._fused_step(vp, g, False)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert bool(torch.isfinite(vp).all())


def test_cholesky_rmsprop_converges(vb):
    """RMSProp on MultivariateT(3, 100, reparam='cholesky') recovers a correlated 3-D Gaussian's mean and covariance
    to one decimal."""
    m = np.array([1.0, -2.0, 0.5])
    C = np.array([[1.0, 0.5, 0.2], [0.5, 2.0, -0.3], [0.2, -0.3, 0.5]])
    np.random.seed(0)
    approx = vb.MultivariateT(3, 100, seed=2, reparam='cholesky')
    obj = vb.ExclusiveKL(approx, _gaussian_model(vb, m, np.linalg.inv(C)), 50)
    res = vb.RMSProp(0.01).optimize(4000, obj, approx.init_param())
    mean, cov = approx.mean_and_cov(res['opt_param'])
    assert np.max(np.abs(mean - m)) < 0.05, mean
    assert np.max(np.abs(cov - C)) < 0.05, cov
