"""CPU: the path-derivative ExclusiveKL of the full-rank MultivariateT (use_path_deriv=True) -- the numpy references of
tests/_mvt_path_ref.py against torch float64 autograd of the reference's expression (objectives.py:156-159): theta
through sqrtm(Sigma(lambda)) (oracle/refshim's sqrtm stand-in) or L(lambda), minus the reference's eigh-based log
density at a detached var_param, mean, backward.  Also the workspace queries of the C ABI."""
import math

import numpy as np
import pytest
import torch

import _mvt_path_ref as pr
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


def _sigma(d, rs, floor):
    """A correlated Sigma with eigenvalues in [0.5, 2]; with floor, one of them is 1e-12, below the 1e-10 floor."""
    Q, R = np.linalg.qr(rs.randn(d, d))
    V = Q * np.sign(np.diag(R))
    w = rs.uniform(0.5, 2.0, d)
    if floor:
        w[0] = 1e-12
    S = (V * w) @ V.T
    return 0.5 * (S + S.T)


def _unpack_t(lam, d):
    rows, cols = np.tril_indices(d)
    F = torch.zeros(d, d, dtype=torch.float64).index_put((torch.as_tensor(rows), torch.as_tensor(cols)), lam[d:])
    return lam[:d], torch.tril(F, -1) + torch.diag(torch.exp(torch.diagonal(F)))


def _t_log_density(vp, x, df):
    """oracle.mvt_log_density (_distributions.py:7-38) in torch, eigenvalue floor included.  vp is detached, so the
    eigen-decomposition is numpy's, the one the numpy reference uses: eigenvalues near 1e-12 carry an absolute error of
    about u |Sigma| that differs between LAPACK drivers, and log w would carry it into the value."""
    from oracle.viabel_oracle import mvt_unpack
    d = x.shape[1]
    mu, L = mvt_unpack(vp.numpy(), d)
    mu = torch.as_tensor(mu)
    w, V = (torch.as_tensor(a) for a in np.linalg.eigh(L @ L.T))
    winv = torch.where(w.abs() <= 1e-10, torch.zeros_like(w), 1.0 / torch.where(w == 0, torch.ones_like(w), w))
    maha = (((x - mu) @ (V * torch.sqrt(winv))) ** 2).sum(dim=-1)
    return (math.lgamma(0.5 * (df + d)) - math.lgamma(0.5 * df) - 0.5 * d * math.log(math.pi * df)
            - 0.5 * torch.log(w).sum() - 0.5 * (df + d) * torch.log(1.0 + maha / df))


def _eigh_sqrtm():
    """oracle/refshim's sqrtm with an eigh forward.  The stand-in's forward is scipy's Schur-method sqrtm, whose error
    of about u |Sigma| / sqrt(w_min) in A is far above the eigh form's when Sigma has an eigenvalue at 1e-12; the
    product and the numpy reference form A from eigh.  The VJP is the stand-in's."""
    from oracle.refshim.autograd.scipy.linalg import _Sqrtm
    from oracle.viabel_oracle import sym_sqrt

    class _EighSqrtm(_Sqrtm):
        @staticmethod
        def forward(ctx, S):
            A = torch.from_numpy(np.ascontiguousarray(sym_sqrt(S.detach().numpy())[0]))
            ctx.save_for_backward(A)
            return A
    return _EighSqrtm


def _autograd_path(vp, chi2, z, df, t_logp, reparam):
    from oracle.refshim.autograd.scipy.linalg import _Sqrtm
    S, d = z.shape
    lam = torch.tensor(vp, dtype=torch.float64, requires_grad=True)
    mu, L = _unpack_t(lam, d)
    zu = torch.as_tensor(z) / torch.sqrt(torch.as_tensor(chi2) / df)[:, None]
    if reparam in ('sqrtm', 'sqrtm-eigh'):
        sqrtm = _Sqrtm if reparam == 'sqrtm' else _eigh_sqrtm()
        theta = mu + zu @ sqrtm.apply(L @ L.T)                  # approximations.py:348
    else:
        theta = mu + zu @ L.T
    value = -(t_logp(theta) - _t_log_density(lam.detach(), theta, df)).mean()
    (g,) = torch.autograd.grad(value, lam)
    return float(value.detach()), g.numpy()


@pytest.mark.parametrize('reparam', ['sqrtm', 'cholesky'])
@pytest.mark.parametrize('d', [3, 12, 40])
def test_oracle_path_gradient_vs_autograd(reparam, d):
    from oracle import viabel_oracle as vo
    df, S = 7.0, 50
    rs = np.random.RandomState(300 + d)
    np_model, t_logp = _target(d, 100 + d)
    vp = vo.mvt_pack(0.3 * rs.randn(d), _sigma(d, rs, False))
    chi2, z = rs.chisquare(df, S), rs.randn(S, d)
    ref = pr.exclusive_kl_mvt_path if reparam == 'sqrtm' else pr.exclusive_kl_mvt_path_cholesky
    v0, g0, _ = ref(vp, chi2, z, np_model, df)
    v1, g1 = _autograd_path(vp, chi2, z, df, t_logp, reparam)
    assert relerr(v0, v1) < TOL64
    assert relerr(g0, g1) < TOL64


@pytest.mark.parametrize('d', [4, 12, 40])
def test_oracle_path_sqrtm_eigenvalue_floor_vs_autograd(d):
    """Sigma with an eigenvalue at 1e-12: the reference's log density drops it from the pseudo-inverse, and so does the
    sqrtm-mode path gradient.  A comes from eigh on both sides (_eigh_sqrtm).  (Eigenvalues 1e-12 and 2e-10 together
    are left to the kernel-level GPU test, where both sides share one eigen-decomposition: their eigenvectors move by
    about u / 2e-10 under the rounding of L L^T, so two decompositions of it cannot agree to 1e-10.)"""
    from oracle import viabel_oracle as vo
    df, S = 7.0, 50
    rs = np.random.RandomState(400 + d)
    np_model, t_logp = _target(d, 500 + d)
    vp = vo.mvt_pack(0.3 * rs.randn(d), _sigma(d, rs, True))
    _, L = vo.mvt_unpack(vp, d)
    w = np.linalg.eigvalsh(L @ L.T)
    assert np.sum(np.abs(w) <= 1e-10) == 1 and np.sum(w < 0.5) == 1
    chi2, z = rs.chisquare(df, S), rs.randn(S, d)
    v0, g0, _ = pr.exclusive_kl_mvt_path(vp, chi2, z, np_model, df)
    v1, g1 = _autograd_path(vp, chi2, z, df, t_logp, 'sqrtm-eigh')
    assert relerr(v0, v1) < TOL64
    assert relerr(g0, g1) < TOL64


def test_path_workspace_queries():
    """The path-derivative form has its own workspace queries; the entropy-form queries keep their sizes."""
    import viabel_b200 as vb
    lib = vb._lib.lib
    S, d = 256, 2048
    assert lib.vb_mvt_chol_path_workspace_bytes(S, d) >= 8 * (2 * d * d + S * d + S)
    assert lib.vb_mvt_chol_objective_workspace_bytes(S, d) < 64 * S * d
    assert lib.vb_mvt_path_workspace_bytes(S, d) >= lib.vb_mvt_objective_workspace_bytes(S, d) + 8 * (2 * S + 3 * d)
    for fn in (lib.vb_mvt_chol_path_workspace_bytes, lib.vb_mvt_path_workspace_bytes):
        assert fn(0, d) == 0 and fn(S, 0) == 0 and fn(-1, d) == 0
