"""numpy float64 references for the path-derivative ExclusiveKL of the full-rank MultivariateT (use_path_deriv=True,
objectives.py:156-159) in both reparameterisations, used by the tests.

    value = -(1/S) sum_s [ f(theta_s) - log q(theta_s) ]   with var_param held fixed in log q (the reference's getval)

and the gradient through theta_s(var_param) only: the entropy-form VJP of each mode with g_s replaced by
g_s - grad_theta log q(theta_s) = g_s + kappa_s y_s, y_s = Sigma^+ (theta_s - mu), kappa_s = (df + d) / (df + delta_s),
delta_s = (theta_s - mu)^T Sigma^+ (theta_s - mu), and no entropy term.  The sqrtm mode applies the reference log
density's eigenvalue floor (_distributions.py:26-28): |w| <= 1e-10 gets a zero inverse.  tests/test_mvt_path_host.py
checks both against torch autograd of the reference's expression.
"""
import math

import numpy as np
from scipy import linalg as sla
from scipy import special as sps

from _mvt_cholesky_ref import _grad, _logq, mvt_sample_cholesky
from oracle.viabel_oracle import _mvt_backprop, mvt_unpack


def _mvt_const(df, d):
    return sps.gammaln(0.5 * (df + d)) - sps.gammaln(0.5 * df) - 0.5 * d * math.log(math.pi * df)


def exclusive_kl_mvt_path(var_param, chi2, z, model, df, w=None, V=None, half_logdet=None):
    """Path-derivative ExclusiveKL with the reference's sqrtm map theta = mu + (z / u) sqrtm(Sigma).  (value, grad, f).

    (w, V) is eigh(Sigma) unless given.  half_logdet replaces the reference's 0.5 sum log w in log q when given (the
    device uses sum_i F_ii, which differs from it by eigh's absolute error in eigenvalues near zero)."""
    S, d = z.shape
    mu, L = mvt_unpack(var_param, d)
    if w is None:
        w, V = np.linalg.eigh(L @ L.T)
    A = (V * np.sqrt(np.maximum(w, 0.0))) @ V.T
    zu = z / np.sqrt(chi2 / df)[:, None]
    theta = mu + zu @ A
    f, g = model(theta)
    winv = np.where(np.abs(w) <= 1e-10, 0.0, 1.0 / np.where(w == 0, 1.0, w))
    R = (theta - mu) @ V
    maha = np.sum(R * R * winv, axis=1)
    y = (R * winv) @ V.T                                       # Sigma^+ (theta - mu), as rows
    if half_logdet is None:
        half_logdet = 0.5 * np.sum(np.log(w))
    logq = _mvt_const(df, d) - half_logdet - 0.5 * (df + d) * np.log(1.0 + maha / df)
    value = -np.mean(f - logq)
    gt = g + ((df + d) / (df + maha))[:, None] * y
    Fbar = _mvt_backprop(-(zu.T @ gt) / S, L, w, V)
    return value, np.concatenate([-np.mean(gt, axis=0), Fbar[np.tril_indices(d)]]), f


def exclusive_kl_mvt_path_cholesky(var_param, chi2, z, model, df):
    """Path-derivative ExclusiveKL with theta = mu + L z / u: y_s = L^-T zhat_s, delta_s = |zhat_s|^2.
    (value, grad, f)."""
    S, d = z.shape
    _, L = mvt_unpack(var_param, d)
    zu = z / np.sqrt(chi2 / df)[:, None]
    f, g = model(mvt_sample_cholesky(var_param, chi2, z, df))
    y = sla.solve_triangular(L, zu.T, lower=True, trans='T').T
    kappa = (df + d) / (df + np.sum(zu * zu, axis=1))
    value = -np.mean(f - _logq(var_param, zu, df))
    return value, _grad(var_param, zu, g + kappa[:, None] * y, np.ones(S), -1.0 / S, 0.0), f
