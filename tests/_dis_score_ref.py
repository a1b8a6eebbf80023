"""Numpy references of the DISInclusiveKL score for the full-rank MultivariateT (csrc/mvt_chol.cu, vb_mvt_score_f64)
and the low-rank LRGaussian (csrc/lr_score.cu, vb_lr_score_f64), independent of the library:

    value = -sum_r c_r log q(x_r; lambda),   grad = d value / d lambda,   c_r = scale * w_r,   x_r = x[idx[r]]

Each takes a dtype: float64, or np.longdouble for the element-wise bounds of the GPU tests.  The long-double path runs
its own triangular and Cholesky solves (numpy's linalg has no long double).  `mutation` drops one term of the gradient
so that the host tests can show the comparison against torch autograd notices it.

MultivariateT (lambda = [mu, tril(F)], L = tril(F,-1) + diag(exp(diag F))):
    y_r = L^-1 (x_r - mu), delta_r = |y_r|^2, kappa_r = (df + d) / (df + delta_r), v_r = L^-T y_r
    gbar_mu = -sum c kappa v,  Fbar_ij = -sum c kappa v_i y_j (j < i),  Fbar_ii = -L_ii sum c kappa v_i y_i + sum c
LRGaussian (lambda = [mu, ls, B]) by Woodbury, M = I + B^T D^-2 B, s_r = Sigma^-1 (x_r - mu):
    gbar_mu = -sum c s,  Bbar = -S^T diag(c) S B + C_tot D^-2 B M^-1,
    lsbar_j = -sigma_j^2 sum c s_j^2 + C_tot (1 - sigma_j^-2 (B M^-1 B^T)_jj)"""
import math

import numpy as np
from scipy.special import gammaln

U64 = 2.0 ** -53
LOG_2PI = math.log(2 * math.pi)


def _rows(x, idx, w, scale, dtype):
    x = np.asarray(x, dtype=dtype)
    rows = x if idx is None else x[np.asarray(idx)]
    n = rows.shape[0]
    c = dtype(scale) * (np.ones(n, dtype=dtype) if w is None else np.asarray(w, dtype=dtype))
    return rows, c


def mvt_unpack(vp, d, dtype=np.float64):
    vp = np.asarray(vp, dtype=dtype)
    F = np.zeros((d, d), dtype=dtype)
    F[np.tril_indices(d)] = vp[d:]
    L = np.tril(F, -1) + np.diag(np.exp(np.diag(F)))
    return vp[:d], F, L


def _lower_solve(L, B):
    """L^-1 B for lower-triangular L (rows of B^T solved together), any dtype"""
    n = L.shape[0]
    X = np.zeros_like(B)
    for i in range(n):
        X[i] = (B[i] - L[i, :i] @ X[:i]) / L[i, i]
    return X


def _upper_solve(Ut, B):
    """Ut^-1 B for upper-triangular Ut, any dtype"""
    n = Ut.shape[0]
    X = np.zeros_like(B)
    for i in reversed(range(n)):
        X[i] = (B[i] - Ut[i, i + 1:] @ X[i + 1:]) / Ut[i, i]
    return X


def _tri_solve(L, B, lower, dtype):
    if dtype == np.float64:
        from scipy.linalg import solve_triangular
        return solve_triangular(L, B, lower=lower)
    return _lower_solve(L, B) if lower else _upper_solve(L, B)


def mvt_score(vp, x, idx, w, scale, df, dtype=np.float64, mutation=None):
    """(value, grad[d + d(d+1)/2], mag) with mag[i] = sum of |summands| of grad[i] (the scale of its rounding)."""
    x = np.asarray(x)
    d = x.shape[1]
    mu, F, L = mvt_unpack(vp, d, dtype)
    rows, c = _rows(x, idx if mutation != 'idx' else None, w, scale, dtype)
    if mutation == 'idx':
        rows, c = rows[:len(idx)], c[:len(idx)]
    D = rows - mu
    Y = _tri_solve(L, D.T, True, dtype).T
    V = _tri_solve(L.T.copy(), Y.T, False, dtype).T
    delta = np.sum(Y * Y, axis=1)
    df_ = dtype(df)
    kappa = (df_ + d) / (df_ + delta)
    if mutation == 'kappa':
        kappa = np.ones_like(kappa)
    const = dtype(gammaln(0.5 * (df + d)) - gammaln(0.5 * df) - 0.5 * d * math.log(math.pi * df))
    lq = const - np.sum(np.diag(F)) - 0.5 * (df_ + d) * np.log1p(delta / df_)
    value = -np.sum(c * lq)
    ck = c * kappa
    gmu = -(ck @ V)
    Fb = -((V * ck[:, None]).T @ Y)
    Fm = np.abs(V * ck[:, None]).T @ np.abs(Y)
    diagL = np.diag(L)
    if mutation != 'chain':
        Fb[np.diag_indices(d)] *= diagL
        Fm[np.diag_indices(d)] *= diagL
    if mutation != 'ctot':
        Fb[np.diag_indices(d)] += np.sum(c)
    Fm[np.diag_indices(d)] += np.sum(np.abs(c))
    grad = np.concatenate([gmu, Fb[np.tril_indices(d)]])
    mag = np.concatenate([np.abs(ck) @ np.abs(V), Fm[np.tril_indices(d)]])
    return value, grad, mag, np.sum(np.abs(c * lq))


def _chol(M):
    """lower Cholesky factor, any dtype"""
    k = M.shape[0]
    C = np.zeros_like(M)
    for j in range(k):
        s = M[j, j] - C[j, :j] @ C[j, :j]
        C[j, j] = np.sqrt(s)
        for i in range(j + 1, k):
            C[i, j] = (M[i, j] - C[i, :j] @ C[j, :j]) / C[j, j]
    return C


def lr_score(vp, x, idx, w, scale, k, dtype=np.float64, mutation=None):
    """(value, grad[2d + d k], mag, value_mag) for LRGaussian, by Woodbury (no projection P)."""
    x = np.asarray(x)
    d = x.shape[1]
    vp = np.asarray(vp, dtype=dtype)
    mu, ls, B = vp[:d], vp[d:2 * d], vp[2 * d:].reshape(d, k)
    sig = np.exp(ls)
    rows, c = _rows(x, idx, w, scale, dtype)
    u = (rows - mu) / sig
    Bd = B / sig[:, None]                                 # D^-1 B
    M = np.eye(k, dtype=dtype) + Bd.T @ Bd
    C = _chol(M)
    t = u @ Bd                                            # (B^T D^-1 u_r) per row
    a = _tri_solve(C, t.T, True, dtype).T                 # C^-1 B^T D^-1 u (= -a_r of the kernel's sign convention)
    Minv_t = _tri_solve(C.T.copy(), a.T, False, dtype).T
    s = (u - Minv_t @ Bd.T) / sig
    logdetM = 2 * np.sum(np.log(np.diag(C))) if k else dtype(0)
    lq = -0.5 * (d * dtype(LOG_2PI) + 2 * np.sum(ls) + logdetM + np.sum(u * u, axis=1) - np.sum(a * a, axis=1))
    value = -np.sum(c * lq)
    ctot = np.sum(c)
    gmu = -(c @ s)
    G = _tri_solve(C, Bd.T, True, dtype)                  # C^-1 B^T D^-1 = -P_B, k x d
    pb2 = np.sum(G * G, axis=0)
    if mutation == 'pb':
        pb2 = np.zeros_like(pb2)
    gls = -sig * sig * (c @ (s * s)) + ctot * (1 - pb2)
    SB = s @ B
    Cinv = _tri_solve(C, np.eye(k, dtype=dtype), True, dtype)
    Bbar = -((s * c[:, None]).T @ SB) + ctot * ((G / sig[None, :]).T @ Cinv)
    grad = np.concatenate([gmu, gls, Bbar.ravel()])
    ac = np.abs(c)
    mag = np.concatenate([ac @ np.abs(s), sig * sig * (ac @ (s * s)) + np.abs(ctot) * (1 + pb2),
                          ((np.abs(s) * ac[:, None]).T @ (np.abs(s) @ np.abs(B)) +
                           np.abs(ctot) * (np.abs(G / sig[None, :]).T @ np.abs(Cinv))).ravel()])
    return value, grad, mag, np.sum(np.abs(c * lq))


def lr_projection(vp, d, k):
    """P = [C^-1 | -C^-1 B^T D^-1] in float64 (what convenience._lr_projection forms on the device)"""
    vp = np.asarray(vp, dtype=np.float64)
    ls, B = vp[d:2 * d], vp[2 * d:].reshape(d, k)
    Bd = B / np.exp(ls)[:, None]
    C = np.linalg.cholesky(np.eye(k) + Bd.T @ Bd)
    from scipy.linalg import solve_triangular
    return solve_triangular(C, np.concatenate([np.eye(k), -Bd.T], axis=1), lower=True)


def mvt_logq_at_draw(vp, zu2, d, df):
    """closed-form log q at a reparameterised draw: const - sum F_ii - (df + d)/2 log1p(|z/u|^2 / df)"""
    vp = np.asarray(vp, dtype=np.float64)
    i = np.arange(d)
    const = gammaln(0.5 * (df + d)) - gammaln(0.5 * df) - 0.5 * d * math.log(math.pi * df)
    return const - np.sum(vp[d + i * (i + 3) // 2]) - 0.5 * (df + d) * np.log1p(zu2 / df)
