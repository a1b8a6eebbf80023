"""numpy float64 reference for MultivariateT's Cholesky reparameterisation (reparam='cholesky'), used by the tests.

theta = mu + L z / u with the L of var_param.  The same distribution as the reference's sqrtm map (L L^T = Sigma), so
the same objectives; the per-draw map, and with it the Monte Carlo gradient, differ.  The gradients are written out
analytically: Fbar = c sum_s sv_s g_s zhat_s^T restricted to the lower triangle, with the chain rule through
L_ii = exp(F_ii) on the diagonal.  tests/test_mvt_cholesky_host.py checks them against torch autograd.
"""
import math

import numpy as np
from scipy import special as sps

from oracle.viabel_oracle import mvt_entropy_stable, mvt_unpack


def mvt_sample_cholesky(var_param, chi2, z, df):
    d = z.shape[1]
    mu, L = mvt_unpack(var_param, d)
    u = np.sqrt(chi2 / df)
    return mu + (z / u[:, None]) @ L.T


def _grad(var_param, zu, g, sv, c, diag_add):
    d = zu.shape[1]
    _, L = mvt_unpack(var_param, d)
    gmu = c * (sv @ g)
    Fbar = np.tril(c * ((sv[:, None] * g).T @ zu))
    Fbar[np.diag_indices(d)] = Fbar[np.diag_indices(d)] * np.diag(L) + diag_add
    return np.concatenate([gmu, Fbar[np.tril_indices(d)]])


def _logq(var_param, zu, df):
    """log q at theta = mu + L zu: the Mahalanobis term is |zu|^2 exactly."""
    d = zu.shape[1]
    _, L = mvt_unpack(var_param, d)
    return (sps.gammaln(0.5 * (df + d)) - sps.gammaln(0.5 * df) - 0.5 * d * math.log(math.pi * df)
            - np.sum(np.log(np.diag(L))) - 0.5 * (df + d) * np.log1p(np.sum(zu * zu, axis=1) / df))


def exclusive_kl_mvt_cholesky(var_param, chi2, z, model, df):
    """ExclusiveKL (entropy branch) with theta = mu + L z / u.  (value, grad, logp)."""
    S, d = z.shape
    zu = z / np.sqrt(chi2 / df)[:, None]
    f, g = model(mvt_sample_cholesky(var_param, chi2, z, df))
    value = -(np.mean(f) + mvt_entropy_stable(var_param, d))
    return value, _grad(var_param, zu, g, np.ones(S), -1.0 / S, -1.0), f


def alpha_divergence_mvt_cholesky(var_param, chi2, z, model, df, alpha):
    """AlphaDivergence with theta = mu + L z / u.  (value, grad, lw)."""
    S, d = z.shape
    zu = z / np.sqrt(chi2 / df)[:, None]
    f, g = model(mvt_sample_cholesky(var_param, chi2, z, df))
    lw = f - _logq(var_param, zu, df)
    m = np.max(lw)
    sv = np.exp(lw - m) ** alpha
    value = np.log(np.mean(sv)) / alpha + m
    return value, _grad(var_param, zu, g, sv, alpha / S, alpha / S * np.sum(sv)), lw
