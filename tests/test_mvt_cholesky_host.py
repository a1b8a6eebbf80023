"""CPU: MultivariateT's Cholesky reparameterisation (theta = mu + L z / u) -- the numpy reference's analytic value and
gradient against torch float64 autograd of the objective written out in full (log q through a triangular solve, not
the |z/u|^2 shortcut the kernels use), the reparam option and the O(S d) workspace of the C ABI."""
import math

import numpy as np
import pytest
import torch

import _mvt_cholesky_ref as cr
from conftest import relerr

TOL64 = 1e-10


def _target(d, seed):
    """Correlated Gaussian target log N(theta; m, P^-1) as a numpy (f, g) model and a torch log density."""
    rs = np.random.RandomState(seed)
    B = rs.randn(d, d) / np.sqrt(d)
    P = np.eye(d) + B @ B.T
    m = rs.randn(d)

    def np_model(theta):
        r = theta - m
        return -0.5 * np.sum((r @ P) * r, axis=1), -r @ P

    Pt, mt = torch.as_tensor(P), torch.as_tensor(m)

    def t_logp(theta):
        r = theta - mt
        return -0.5 * ((r @ Pt) * r).sum(dim=1)
    return np_model, t_logp


def _point(d, df, S, seed):
    from oracle import viabel_oracle as vo
    rs = np.random.RandomState(seed)
    B = 0.4 * rs.randn(d, d) / np.sqrt(d)
    vp = vo.mvt_pack(0.3 * rs.randn(d), 0.5 * np.eye(d) + B @ B.T)
    return vp, rs.chisquare(df, S), rs.randn(S, d)


def _autograd(vp, chi2, z, df, t_logp, alpha):
    """(value, grad) by autograd; alpha None = ExclusiveKL (entropy form), else AlphaDivergence's surrogate
    alpha * mean(sv.detach() * lw) (objectives.py:443-460)."""
    S, d = z.shape
    lam = torch.tensor(vp, dtype=torch.float64, requires_grad=True)
    mu = lam[:d]
    rows, cols = np.tril_indices(d)
    F = torch.zeros(d, d, dtype=torch.float64).index_put((torch.as_tensor(rows), torch.as_tensor(cols)), lam[d:])
    L = torch.tril(F, -1) + torch.diag(torch.exp(torch.diagonal(F)))
    zu = torch.as_tensor(z) / torch.sqrt(torch.as_tensor(chi2) / df)[:, None]
    theta = mu + zu @ L.T
    f = t_logp(theta)
    if alpha is None:
        value = -(f.mean() + torch.diagonal(F).sum())
        (g,) = torch.autograd.grad(value, lam)
        return float(value.detach()), g.numpy()
    # multivariate t log density of theta under (mu, L L^T), Mahalanobis term by a triangular solve
    y = torch.linalg.solve_triangular(L, (theta - mu).T, upper=False)
    maha = (y * y).sum(dim=0)
    logq = (math.lgamma(0.5 * (df + d)) - math.lgamma(0.5 * df) - 0.5 * d * math.log(math.pi * df)
            - torch.diagonal(F).sum() - 0.5 * (df + d) * torch.log1p(maha / df))
    lw = f - logq
    m = lw.max().detach()
    sv = torch.exp(lw - m) ** alpha
    (g,) = torch.autograd.grad(alpha * (sv.detach() * lw).mean(), lam)
    return float(torch.log(sv.mean()).detach() / alpha + m), g.numpy()


@pytest.mark.parametrize('d', [3, 12, 40])
@pytest.mark.parametrize('alpha', [None, 1.5, 2.0])
def test_oracle_cholesky_gradient_vs_autograd(d, alpha):
    from oracle import viabel_oracle as vo
    df, S = 7.0, 50
    np_model, t_logp = _target(d, 100 + d)
    vp, chi2, z = _point(d, df, S, 200 + d)
    if alpha is None:
        v0, g0, _ = cr.exclusive_kl_mvt_cholesky(vp, chi2, z, np_model, df)
    else:
        v0, g0, _ = cr.alpha_divergence_mvt_cholesky(vp, chi2, z, np_model, df, alpha)
    v1, g1 = _autograd(vp, chi2, z, df, t_logp, alpha)
    assert relerr(v0, v1) < TOL64
    assert relerr(g0, g1) < TOL64


def test_oracle_cholesky_sample_matches_covariance():
    """L L^T = Sigma: the Cholesky map of z is a linear map with the sqrtm map's covariance."""
    from oracle import viabel_oracle as vo
    d, df = 6, 9.0
    vp, _, _ = _point(d, df, 1, 5)
    mu, L = vo.mvt_unpack(vp, d)
    ones = np.full(d, df)
    x = cr.mvt_sample_cholesky(vp, ones, np.eye(d), df) - mu          # rows: L e_k
    y = vo.mvt_sample(vp, ones, np.eye(d), df) - mu                     # rows: sqrtm(Sigma) e_k
    assert relerr(x.T @ x, y.T @ y) < 1e-12


def test_invalid_reparam_raises():
    import viabel_b200 as vb
    with pytest.raises(ValueError):
        vb.MultivariateT(4, 10.0, reparam='eigh')
    with pytest.raises(ValueError):
        vb.MultivariateT(4, 10.0, reparam=None)
    assert vb.MultivariateT(4, 10.0).reparam == 'sqrtm'
    assert vb.MultivariateT(4, 10.0, reparam='cholesky').reparam == 'cholesky'


def test_cholesky_workspace_is_O_S_d():
    import viabel_b200 as vb
    S, d = 256, 2048
    nbytes = vb._lib.lib.vb_mvt_chol_objective_workspace_bytes(S, d)
    assert 0 < nbytes < 64 * S * d
    assert vb._lib.lib.vb_mvt_chol_objective_workspace_bytes(0, d) == 0
