"""CPU checks of the DISInclusiveKL score references (tests/_dis_score_ref.py) against torch autograd of the
reference's own log densities: the eigh-based multivariate_t_logpdf with its 1e-10 floor (_distributions.py:7-38) for
MultivariateT and a dense-Sigma Gaussian log density for LRGaussian.  Also records that autograd through eigh is not
finite at the family's init point Sigma = 10 I, where the analytic gradient is, and that dropping any one term of the
analytic gradient is caught by the comparison."""
import math

import numpy as np
import pytest
import torch

import _dis_score_ref as R


def _mvt_point(d, cond, rs):
    """var_param whose Sigma = L L^T has distinct eigenvalues spanning about `cond`"""
    Q, _ = np.linalg.qr(rs.randn(d, d))
    ev = np.logspace(0, math.log10(cond), d) * (1 + 0.01 * np.arange(d))
    Sigma = (Q * ev) @ Q.T
    L = np.linalg.cholesky(Sigma)
    F = np.tril(L, -1) + np.diag(np.log(np.diag(L)))
    return np.concatenate([rs.randn(d), F[np.tril_indices(d)]])


def _mvt_logpdf_t(lam, x, d, df):
    """multivariate_t_logpdf as the reference writes it: eigh of Sigma, floored pseudo-inverse"""
    mu = lam[:d]
    F = torch.zeros(d, d, dtype=torch.float64)
    F[tuple(torch.tril_indices(d, d))] = lam[d:]
    L = torch.tril(F, -1) + torch.diag(torch.exp(torch.diagonal(F)))
    w, V = torch.linalg.eigh(L @ L.T)
    winv = torch.where(w.abs() <= 1e-10, torch.zeros_like(w), 1.0 / w)
    maha = ((((x - mu) @ V) ** 2) * winv).sum(dim=1)
    c = math.lgamma(0.5 * (df + d)) - math.lgamma(0.5 * df) - 0.5 * d * math.log(math.pi * df)
    return c - 0.5 * torch.log(w).sum() - 0.5 * (df + d) * torch.log1p(maha / df)


def _autograd_score(logpdf, vp, x, idx, w, scale):
    lam = torch.tensor(vp, dtype=torch.float64, requires_grad=True)
    xs = torch.tensor(x if idx is None else x[idx], dtype=torch.float64)
    c = scale * (torch.ones(xs.shape[0], dtype=torch.float64) if w is None else torch.tensor(w))
    value = -(c * logpdf(lam, xs)).sum()
    (g,) = torch.autograd.grad(value, lam)
    return float(value.detach()), g.numpy()


def _relerr(a, b):
    return np.linalg.norm(np.asarray(a) - np.asarray(b)) / np.linalg.norm(b)


def _mvt_case(d, cond, seed):
    rs = np.random.RandomState(seed)
    vp = _mvt_point(d, cond, rs)
    x = rs.randn(20, d) * 2 + vp[:d]
    idx = np.array([3, 3, 17, 0, 9, 3, 12])
    w = rs.rand(len(idx)) + 0.1
    return vp, x, idx, w, 0.37


@pytest.mark.parametrize('d,cond', [(3, 10.0), (3, 1e6), (7, 1e3), (7, 1e6)])
@pytest.mark.parametrize('df', [3.5, 100.0])
def test_mvt_score_matches_autograd(d, cond, df):
    vp, x, idx, w, scale = _mvt_case(d, cond, 11 * d)
    v0, g0 = _autograd_score(lambda lam, xs: _mvt_logpdf_t(lam, xs, d, df), vp, x, idx, w, scale)
    v, g, _, _ = R.mvt_score(vp, x, idx, w, scale, df)
    # the eigh route rounds at about cond * u (its backward also divides by eigenvalue gaps)
    tol = 1e-12 if cond < 1e4 else 1e-8
    assert abs(v - v0) <= tol * abs(v0)
    assert _relerr(g, g0) < tol, _relerr(g, g0)
    vl, gl, _, _ = R.mvt_score(vp, x, idx, w, scale, df, dtype=np.longdouble)
    assert _relerr(g, gl.astype(np.float64)) < 1e-12


def test_mvt_eigh_gradient_not_finite_at_init():
    """At Sigma = 10 I (the family's init_param) autograd through eigh divides by zero eigenvalue gaps; the analytic
    score gradient is the finite gradient of the same smooth function, which a finite difference confirms."""
    d, df = 3, 5.0
    F = np.diag(np.full(d, 0.5 * np.log(10.0)))
    vp = np.concatenate([np.zeros(d), F[np.tril_indices(d)]])
    x = np.random.RandomState(0).randn(6, d)
    _, g0 = _autograd_score(lambda lam, xs: _mvt_logpdf_t(lam, xs, d, df), vp, x, None, None, 1.0)
    assert not np.all(np.isfinite(g0))
    v, g, _, _ = R.mvt_score(vp, x, None, None, 1.0, df)
    assert np.all(np.isfinite(g))
    h = 1e-6
    for i in range(vp.size):
        e = np.zeros(vp.size)
        e[i] = h
        fd = (R.mvt_score(vp + e, x, None, None, 1.0, df)[0] - R.mvt_score(vp - e, x, None, None, 1.0, df)[0]) / (2 * h)
        assert abs(fd - g[i]) < 1e-6 * max(1.0, abs(g[i]))


@pytest.mark.parametrize('mutation', ['ctot', 'chain', 'kappa', 'idx'])
def test_mvt_mutations_are_caught(mutation):
    d, df = 7, 4.0
    vp, x, idx, w, scale = _mvt_case(d, 1e3, 5)
    _, g0 = _autograd_score(lambda lam, xs: _mvt_logpdf_t(lam, xs, d, df), vp, x, idx, w, scale)
    _, g, _, _ = R.mvt_score(vp, x, idx, w, scale, df, mutation=mutation)
    assert _relerr(g, g0) > 1e-3


def _lr_logpdf_t(lam, x, d, k):
    mu, ls, B = lam[:d], lam[d:2 * d], lam[2 * d:].reshape(d, k)
    Sigma = B @ B.T + torch.diag(torch.exp(2 * ls))
    diff = x - mu
    maha = (diff * torch.linalg.solve(Sigma, diff.T).T).sum(dim=1)
    return -0.5 * (d * math.log(2 * math.pi) + torch.linalg.slogdet(Sigma)[1] + maha)


def _lr_case(d, k, seed):
    rs = np.random.RandomState(seed)
    vp = np.concatenate([rs.randn(d), 0.3 * rs.randn(d), rs.randn(d * k)])
    x = rs.randn(15, d) * 2
    idx = np.array([14, 2, 2, 7, 0, 2])
    w = rs.rand(len(idx)) + 0.1
    return vp, x, idx, w, 0.61


@pytest.mark.parametrize('k', [0, 1, 3])
@pytest.mark.parametrize('d', [3, 7])
def test_lr_score_matches_autograd(d, k):
    vp, x, idx, w, scale = _lr_case(d, k, 3 * d + k)
    v0, g0 = _autograd_score(lambda lam, xs: _lr_logpdf_t(lam, xs, d, k), vp, x, idx, w, scale)
    v, g, _, _ = R.lr_score(vp, x, idx, w, scale, k)
    assert abs(v - v0) <= 1e-12 * abs(v0)
    assert _relerr(g, g0) < 1e-12, _relerr(g, g0)
    vl, gl, _, _ = R.lr_score(vp, x, idx, w, scale, k, dtype=np.longdouble)
    assert _relerr(g, gl.astype(np.float64)) < 1e-12


def test_lr_mutation_is_caught():
    d, k = 7, 3
    vp, x, idx, w, scale = _lr_case(d, k, 1)
    _, g0 = _autograd_score(lambda lam, xs: _lr_logpdf_t(lam, xs, d, k), vp, x, idx, w, scale)
    _, g, _, _ = R.lr_score(vp, x, idx, w, scale, k, mutation='pb')
    assert _relerr(g, g0) > 1e-3


def test_lr_projection_gives_the_woodbury_terms():
    """the projection the kernel takes: |u|^2 - |P u|^2 is the Mahalanobis term and P_B's column norms the ls term"""
    d, k = 7, 3
    vp, x, _, _, _ = _lr_case(d, k, 2)
    P = R.lr_projection(vp, d, k)
    ls, B = vp[d:2 * d], vp[2 * d:].reshape(d, k)
    Sigma = B @ B.T + np.diag(np.exp(2 * ls))
    u = (x - vp[:d]) / np.exp(ls)
    full = np.concatenate([np.zeros((x.shape[0], k)), u], axis=1)
    maha = np.sum(u * u, axis=1) - np.sum((full @ P.T) ** 2, axis=1)
    np.testing.assert_allclose(maha, np.sum((x - vp[:d]) * np.linalg.solve(Sigma, (x - vp[:d]).T).T, axis=1), rtol=1e-12)
    np.testing.assert_allclose(np.sum(P[:, k:] ** 2, axis=0), 1 - np.exp(2 * ls) * np.diag(np.linalg.inv(Sigma)),
                               rtol=1e-10)
