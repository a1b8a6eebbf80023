"""numpy restatement of the fused AlphaDivergence step (csrc/engine.cu, VB_OBJ_ALPHA), independent of the library.

The step never forms the per-sample model gradients the oracle multiplies by the weights.  It splits the model into
the GLM likelihood, whose weighted sums come out of the second sweep, and the iid Gaussian prior, whose part it forms
from per-column sums of the draws (SURVEY.md App. A.2):

    lw_s  = ll_s + log prior(theta_s) - log q(theta_s),   m = max lw,   w_s = exp(lw_s - m) ** alpha
    value = log(mean w) / alpha + m
    a_j   = sum_s w_s g_sj - (sum_s w_s theta_sj) / tau^2                     (g: likelihood gradient)
    b_j   = sum_s w_s g_sj e_sj - (sum_s w_s theta_sj e_sj) / tau^2
    grad  = (alpha / S) [a,  b sigma + sum_s w_s]

`alpha_step` computes exactly that; tests/test_alpha_step_host.py checks it against the oracle.  `alpha_loop` is the
reference loop of the fused optimise step: oracle value and gradient, then the oracle's RMSProp / Adam update."""
import numpy as np
from scipy import special


def logistic_ll_grad(theta, X, y):
    """likelihood part of the logistic GLM plugin (no prior): ll[S], g[S, d]"""
    z = (theta @ X.T) * y[None, :]                      # [S, N]
    ll = -np.sum(np.logaddexp(0.0, -z), axis=1)
    r = special.expit(-z) * y[None, :]
    return ll, r @ X


def alpha_step(var_param, base, X, y, prior_sd, alpha, family='gaussian', df=None):
    """(value, grad, lw) of one AlphaDivergence evaluation in the fused step's decomposition"""
    S, d = base.shape
    mu, ls = var_param[:d], var_param[d:]
    sig = np.exp(ls)
    theta = mu + sig * base
    ll, g = logistic_ll_grad(theta, X, y)
    prior = -0.5 * np.sum(theta ** 2, axis=1) / prior_sd ** 2 - d * np.log(prior_sd * np.sqrt(2 * np.pi))
    if family == 'gaussian':
        logq = np.sum(-0.5 * base ** 2 - ls - 0.5 * np.log(2 * np.pi), axis=1)
    else:
        tconst = special.gammaln(0.5 * (df + 1)) - special.gammaln(0.5 * df) - 0.5 * np.log(np.pi * df)
        logq = np.sum(tconst - 0.5 * (df + 1) * np.log1p(base ** 2 / df) - ls, axis=1)
    lw = ll + prior - logq
    m = np.max(lw)
    w = np.exp(lw - m) ** alpha
    value = np.log(np.mean(w)) / alpha + m
    a = w @ g - (w @ theta) / prior_sd ** 2
    b = w @ (g * base) - (w @ (theta * base)) / prior_sd ** 2
    grad = alpha / S * np.concatenate([a, b * sig + np.sum(w)])
    return value, grad, lw


def alpha_loop(vo, vp, bases, model, alpha, opt, family='gaussian', df=None, lr=0.01):
    """[(value, grad, var_param after the update)] of the reference loop on the given draws"""
    state = {}
    out = []
    for base in bases:
        v, g, _ = vo.alpha_divergence_meanfield(vp, base, model, alpha, family, df)
        dd = vo.rmsprop_direction(state, g) if opt == 'rmsprop' else vo.adam_direction(state, g)
        vp = vp - lr * dd
        out.append((v, g, vp.copy()))
    return out
