"""Extended-precision reference and worst-case error model of the unfused mean-field kernels (csrc/mf.cu, targets.cu,
opt.cu, dis.cu), independent of the library.

Each function restates one C entry point on float64 inputs in long double (mpmath where long double carries fewer than
64 mantissa bits, through _philox_ref) and returns, next to each output, a bound on the device's float64 error:

    |dev - ref| <= C u (n_chain sum|summands| + sum of the per-term budgets)

n_chain is the longest chain of roundings in the kernel's own summation order (the lane-strided loop plus five shuffle
levels, the 8 or 32 row groups, the block shares).  The per-term budgets use CUDA's documented bounds: exp, log and
log1p 1 ulp, pow 2 ulp (1 ulp <= 2u |x|); + - * / and sqrt are correctly rounded.  A device value outside its bound is
a wrong value, not rounding.  Where exp(lw - m) of the alpha weights is subnormal or zero the bound is absolute: the
float64 quantum 2^-1074 carried through pow.

The DIS bisection reference (objectives.py:317-366) records, for each of its rounds, the margin |ESS - target| over
the ESS error bound: where every margin is above one the device must take the same branch in every round and return
the same epsilon bit for bit; otherwise its epsilon can only be placed within the interval still open at the first
round whose margin is not."""
import math

import mpmath
import numpy as np

import _philox_ref as pr
from _philox_ref import U, abs64, to64, xf

C = 2.0                                  # margin on the worst-case bounds
Q = 2.0 ** -1074                         # float64 subnormal quantum
GAUSS, STUDENT = 0, 1
EKL, EKL_PATH, ALPHA = 0, 1, 2
_exp, _log, _log1p, _pow = pr._exp, pr._log, pr._log1p, pr._pow


def _xconst(x):
    """an mpmath value in extended precision (float64 head + tail)"""
    hi = float(x)
    return xf(hi) + xf(float(x - hi))


def log_t_const(df):
    """log Gamma((df + 1) / 2) - log Gamma(df / 2) - log(pi df) / 2, from mpmath at 120 bits"""
    with mpmath.workprec(120):
        df = mpmath.mpf(df)
        return _xconst(mpmath.loggamma((df + 1) / 2) - mpmath.loggamma(df / 2) - mpmath.log(mpmath.pi * df) / 2)


def _t_const_err(df):
    """error of the host's float64 lgamma((df+1)/2) - lgamma(df/2) - log(pi df)/2 (glibc lgamma within a few ulp)"""
    return U * (8 * (abs(math.lgamma(0.5 * (df + 1))) + abs(math.lgamma(0.5 * df))) + 6 * abs(0.5 * math.log(math.pi * df)))


with mpmath.workprec(120):
    LOG_2PI = _xconst(mpmath.log(2 * mpmath.pi))


def lanes(d):
    """chain of a warp-per-row sum over d columns: the lane-strided loop plus five shuffle levels"""
    return -(-d // 32) + 5


def ratio(dev, ref, bound):
    """largest |dev - ref| / bound (a NaN or an infinite device value where the reference is finite: inf)"""
    dev = np.asarray(dev, dtype=np.float64)
    e = pr.err64(dev, ref)
    e = np.where(np.isfinite(dev), e, np.inf)
    b = np.asarray(bound, dtype=np.float64)
    with np.errstate(divide='ignore', invalid='ignore', over='ignore'):
        r = np.where(e == 0, 0.0, e / b)
    return float(np.max(r)) if r.size else 0.0


def _a(x):
    return abs64(x)


# ---- mean-field log density term ----------------------------------------------------------------------------------
def _q_term(z, zrel, ls, family, df):
    """log q per coordinate at standardised z (relative error zrel in float64) and its per-term error budget"""
    lsx = xf(ls)
    if family == GAUSS:
        h = 0.5 * z * z
        t = -h - lsx - 0.5 * LOG_2PI
        budget = U * ((2 * zrel / U + 1) * _a(h) + 2 * (_a(h) + np.abs(ls) + 0.92))
        return t, budget
    tc = log_t_const(df)
    x = z * z / df
    L = _log1p(x)
    h = 0.5 * (df + 1.0)
    t = tc - h * L - lsx
    xa, La = _a(x), _a(L)
    xrel = 2 * zrel + 2 * U
    budget = (h * (xa / (1 + xa) * xrel + 2 * U * La) + 2 * U * h * La + _t_const_err(df)
              + 2 * U * (abs(float(tc)) + h * La + np.abs(ls)))
    return t, budget


# ---- vb_mf_sample_f64 --------------------------------------------------------------------------------------------
def sample(vp, base):
    d = base.shape[1]
    mu, ls = vp[:d], vp[d:]
    se = _exp(xf(ls)) * xf(base)
    th = xf(mu) + se
    return th, C * U * (3 * _a(se) + _a(th))


# ---- vb_mf_log_density_f64 ---------------------------------------------------------------------------------------
def log_density(vp, x, family, df):
    d = x.shape[1]
    mu, ls = vp[:d], vp[d:]
    z = (xf(x) - xf(mu)) / _exp(xf(ls))
    t, budget = _q_term(z, 4 * U, ls, family, df)
    out = t.sum(axis=1)
    return out, C * (U * lanes(d) * _a(t).sum(axis=1) + budget.sum(axis=1))


# ---- vb_target_logp_grad_f64 -------------------------------------------------------------------------------------
def target_logp_grad(theta, kind, loc, scale, df, cst):
    S, d = theta.shape
    sc = xf(scale)
    z = (xf(theta) - xf(loc)) / sc
    if kind == 0:
        t = -0.5 * z * z
        budget = 6 * U * _a(t)
        g = -z / sc
        grel = 4 * U
    else:
        x = z * z / df
        L = _log1p(x)
        h = 0.5 * (df + 1.0)
        t = -h * L
        xa = _a(x)
        budget = h * (xa / (1 + xa) * 6 * U + 2 * U * _a(L)) + 2 * U * _a(t)
        g = -(df + 1.0) * z / ((df + z * z) * sc)
        grel = 13 * U
    lp = t.sum(axis=1)
    lpb = U * lanes(d) * _a(t).sum(axis=1) + budget.sum(axis=1)
    lp = lp + cst
    lpb = lpb + U * (_a(lp) + abs(cst))
    return lp, C * lpb, g, C * grel * _a(g)


# ---- vb_mf_reduce_grads_f64 --------------------------------------------------------------------------------------
def reduce_grads(G, w, e):
    S, d = G.shape
    wx = xf(np.ones(S) if w is None else w)[:, None]
    g = wx * xf(G)
    ge = g * xf(e)
    n = -(-S // 8) + 8
    return (g.sum(axis=0), C * U * (n + 1) * _a(g).sum(axis=0),
            ge.sum(axis=0), C * U * (n + 1) * _a(ge).sum(axis=0))


# ---- per-sample prior and log q (sample_terms) -------------------------------------------------------------------
def _prior_consts(prior_sd, d):
    """(inv_tau2, prior_const) exact, and their float64 errors on the host"""
    if prior_sd > 0 and np.isfinite(prior_sd):
        sd = xf(prior_sd)
        it = 1 / (sd * sd)
        pc = -d * _log(sd * pr._sqrt(2 * pr._PI))
        return it, pc, 2 * U * float(it), U * (3 * abs(float(pc)) + 4 * d)
    return xf(0.0), xf(0.0), 0.0, 0.0


def _terms(vp, theta, base, family, df, prior_sd, want_logq=True):
    """prior_s, its error, logq_s (at z = base), its error"""
    S, d = theta.shape
    n = lanes(d)
    th = xf(theta)
    sq = (th * th).sum(axis=1)
    sq_err = U * (n + 1) * _a(sq)
    it, pc, it_err, pc_err = _prior_consts(prior_sd, d)
    prior = -0.5 * sq * it + pc
    prior_err = (0.5 * float(it) * sq_err + 0.5 * _a(sq) * (it_err + 2 * U * float(it)) + pc_err
                 + U * (_a(prior) + _a(0.5 * sq * it)))
    if not want_logq:
        return prior, prior_err, None, None
    t, budget = _q_term(xf(base), 0.0, np.broadcast_to(vp[d:], base.shape), family, df)
    lq = t.sum(axis=1)
    lq_err = U * n * _a(t).sum(axis=1) + budget.sum(axis=1)
    return prior, prior_err, lq, lq_err


# ---- vb_mf_alpha_weights_f64 -------------------------------------------------------------------------------------
def log_weights(vp, theta, base, ll, family, df, prior_sd):
    prior, prior_err, lq, lq_err = _terms(vp, theta, base, family, df, prior_sd)
    lw = xf(ll) + prior - lq
    return lw, C * (prior_err + lq_err + 2 * U * (np.abs(ll) + _a(prior) + _a(lq)))


def alpha_weights(lw, alpha, m=None):
    """w and value from float64 log-weights lw (the device's own, checked separately): w = exp(lw - m)^alpha,
    value = log(mean w) / alpha + m.  `m` overrides the maximum."""
    lw = np.asarray(lw, dtype=np.float64)
    S = lw.size
    m = float(np.max(lw)) if m is None else m
    r = xf(lw) - xf(m)
    v0 = _exp(r)
    w = _pow(v0, xf(alpha))
    wa = _a(w)
    # relative: pow 2 ulp, alpha x (exp 1 ulp + the rounded difference); absolute: the subnormal quantum of exp(r)
    # carried through pow, and pow's own 2 ulp of a subnormal result
    quantum = _a(_pow(v0 + 2 * Q, xf(alpha)) - w) + 4 * Q
    w_err = wa * (4 * U + alpha * (2 * U + U * _a(r))) + quantum
    acc = w.sum()
    n = -(-S // 1024) + 10
    acc_err = U * n * float(wa.sum()) + float(w_err.sum())
    la = _log(acc / S)
    value = la / alpha + m
    val_err = (acc_err / float(acc) + 3 * U + 2 * U * abs(float(la))) / alpha + U * (abs(float(la / alpha)) + abs(float(value)))
    return w, C * w_err, value, C * val_err


# ---- vb_mf_objective_finish_f64: value and logp -------------------------------------------------------------------
def entropy(vp, d, family):
    ls = xf(vp[d:])
    H = ls.sum()
    err = U * (-(-d // 256) + 10) * float(np.abs(vp[d:]).sum())
    if family == GAUSS:
        H = H + 0.5 * d * (1 + LOG_2PI)
        err += U * 3 * 0.5 * d * 2.84
    return H, err + U * abs(float(H))


def value_terms(vp, theta, base, ll, family, df, prior_sd, objective):
    """per-sample summands acc_s of the ExclusiveKL value (f or f - log q), their errors, and f = logp"""
    path = objective == EKL_PATH
    prior, prior_err, lq, lq_err = _terms(vp, theta, base, family, df, prior_sd, want_logq=path)
    f = xf(ll) + prior
    f_err = prior_err + U * _a(f)
    if not path:
        return f, f_err, f, f_err
    acc = f - lq
    return acc, f_err + lq_err + U * _a(acc), f, f_err


def value_from_terms(acc, acc_err, vp, d, family, objective):
    """value = -(sum_s acc_s / S + H): 8 samples per block (block_sum), one share per block, the shares summed by one
    256-thread block"""
    S = acc.shape[0]
    H, H_err = (entropy(vp, d, family) if objective == EKL else (xf(0.0), 0.0))
    value = -(acc.sum() / S + H)
    nb = -(-S // 8)
    n = 10 + 2 + (-(-nb // 256)) + 10
    err = U * n * (float(_a(acc).sum()) / S + abs(float(H))) + float(np.sum(acc_err)) / S + H_err + U * abs(float(value))
    return value, C * err


def value_and_logp(vp, theta, base, ll, family, df, prior_sd, objective):
    d = theta.shape[1]
    acc, acc_err, f, f_err = value_terms(vp, theta, base, ll, family, df, prior_sd, objective)
    value, verr = value_from_terms(acc, acc_err, vp, d, family, objective)
    return value, verr, f, C * f_err


# ---- vb_mf_objective_finish_f64: gradient -------------------------------------------------------------------------
def grad_pieces(vp, theta, base, w, family, df, objective):
    """the column sums of mf_grad_kernel (p1, p2, pa, pb, sw) and their error bounds; 8 row groups"""
    S, d = theta.shape
    n = -(-S // 8) + 8
    wx = xf(np.ones(S) if w is None else w)[:, None]
    th, e = xf(theta), xf(base)
    t1, t2 = wx * th, wx * th * e
    P = {'p1': t1.sum(axis=0), 'p2': t2.sum(axis=0), 'sw': np.broadcast_to(wx, (S, d)).sum(axis=0)}
    E = {'p1': U * (n + 1) * _a(t1).sum(axis=0), 'p2': U * (n + 2) * _a(t2).sum(axis=0),
         'sw': U * n * _a(np.broadcast_to(wx, (S, d))).sum(axis=0)}
    if objective == EKL_PATH:
        if family == GAUSS:
            ta, tb, ra, rb = e, e * e, 0.0, U
        else:
            q = (df + 1.0) / (df + e * e)
            ta, tb, ra, rb = q * e, q * e * e, 6 * U, 7 * U
        P['pa'], P['pb'] = ta.sum(axis=0), tb.sum(axis=0)
        E['pa'] = U * n * _a(ta).sum(axis=0) + ra * _a(ta).sum(axis=0)
        E['pb'] = U * n * _a(tb).sum(axis=0) + rb * _a(tb).sum(axis=0)
    return P, E


def grad_assemble(P, E, vp, gmu, ge, prior_sd, objective, alpha, S):
    d = gmu.shape[0]
    it, _, it_err, _ = _prior_consts(prior_sd, d)
    itf = float(it)
    sig = _exp(xf(vp[d:]))
    sa = _a(sig)
    inv = 1 / xf(float(S))
    a = xf(gmu) - P['p1'] * it
    b = xf(ge) - P['p2'] * it
    ea = E['p1'] * itf + _a(P['p1']) * (it_err + U * itf) + U * _a(a)
    eb = E['p2'] * itf + _a(P['p2']) * (it_err + U * itf) + U * _a(b)
    bs = b * sig
    ebs = eb * sa + 3 * U * _a(bs)
    if objective == EKL:
        g1 = -inv * a
        g2 = -inv * bs - 1.0
        e1 = ea / S + 2 * U * _a(g1)
        e2 = ebs / S + 2 * U * _a(bs) / S + U * _a(g2)
    elif objective == EKL_PATH:
        s1 = a + P['pa'] / sig
        s2 = bs + P['pb']
        g1, g2 = -inv * s1, -inv * s2
        e1 = (ea + E['pa'] / sa + 3 * U * _a(P['pa'] / sig) + U * _a(s1)) / S + 2 * U * _a(g1)
        e2 = (ebs + E['pb'] + U * _a(s2)) / S + 2 * U * _a(g2)
    else:
        s2 = bs + P['sw']
        g1, g2 = alpha * inv * a, alpha * inv * s2
        e1 = alpha * ea / S + 3 * U * _a(g1)
        e2 = alpha * (ebs + E['sw'] + U * _a(s2)) / S + 3 * U * _a(g2)
    return np.concatenate([g1, g2]), C * np.concatenate([e1, e2])


def grad(vp, theta, base, gmu, ge, w, family, df, prior_sd, objective, alpha):
    P, E = grad_pieces(vp, theta, base, w if objective == ALPHA else None, family, df, objective)
    return grad_assemble(P, E, vp, gmu, ge, prior_sd, objective, alpha, theta.shape[0])


# ---- vb_mf_score_f64 ---------------------------------------------------------------------------------------------
def score(vp, x, idx, w, scale, family, df):
    """value = -sum_r c_r log q(x_idx[r]), grad wrt [mu, log sigma]; c_r = scale w[r]; 32 row groups per column"""
    d = x.shape[1]
    rows = np.arange(x.shape[0]) if idx is None else np.asarray(idx)
    n = rows.size
    mu, ls = vp[:d], vp[d:]
    sig = _exp(xf(ls))
    c = xf(scale) * (xf(np.ones(n)) if w is None else xf(w))[:, None]
    z = (xf(x[rows]) - xf(mu)) / sig
    lq, lq_budget = _q_term(z, 4 * U, np.broadcast_to(ls, z.shape), family, df)
    if family == GAUSS:
        dmu, dls = z / sig, z * z - 1
        emu, els = 9 * U * _a(dmu), 9 * U * _a(z * z) + 3 * U * _a(dls)
    else:
        q = (df + 1.0) / (df + z * z)
        dmu, dls = q * z / sig, q * z * z - 1
        emu, els = 22 * U * _a(dmu), 22 * U * _a(q * z * z) + 3 * U * _a(dls)
    ca = _a(c)
    tv, tm, tl = c * lq, c * dmu, c * dls
    nr = -(-n // 32) + 32
    nb = -(-d // 32)
    gm = -tm.sum(axis=0)
    gl = -tl.sum(axis=0)
    egm = U * nr * _a(tm).sum(axis=0) + (ca * emu).sum(axis=0) + U * _a(tm).sum(axis=0)
    egl = U * nr * _a(tl).sum(axis=0) + (ca * els).sum(axis=0) + U * _a(tl).sum(axis=0)
    value = -tv.sum()
    ev = U * (nr + 10 + nb) * float(_a(tv).sum()) + float((ca * lq_budget).sum()) + 2 * U * float(_a(tv).sum())
    return value, C * ev, np.concatenate([gm, gl]), C * np.concatenate([egm, egl])


# ---- vb_rmsprop_step_f64 / vb_adam_step_f64 ----------------------------------------------------------------------
def rmsprop(vp, g, nu, lr, beta, jitter, first):
    """(vp_new, nu_new, direction) and their bounds (optimization.py:188-197)"""
    gx = xf(g)
    g2 = gx * gx
    v0 = g2 if first else xf(nu)
    v = v0 * beta + (1 - beta) * g2
    ev = U * (3 * _a(v0 * beta) + 4 * _a((1 - beta) * g2) + _a(v))
    return _step_out(vp, gx, _a(gx) * 0, v, ev, lr, jitter)


def adam(vp, g, m, nu, lr, beta1, beta2, jitter, first):
    """(vp_new, m_new, nu_new, direction) and bounds (optimization.py:308-326, the first-step aliasing included)"""
    gx = xf(g)
    if first:
        gs = gx * beta1
        mi = gs + (1 - beta1) * gs
        em = U * (2 * _a(gs) + 3 * _a((1 - beta1) * gs) + _a(mi))
        vi = gx * gx * beta2 + (1 - beta2) * mi * mi
        ev = U * (3 * _a(gx * gx * beta2) + 4 * _a((1 - beta2) * mi * mi) + _a(vi)) + 2 * _a((1 - beta2) * mi) * em
    else:
        mi = xf(m) * beta1 + (1 - beta1) * gx
        em = U * (2 * _a(xf(m) * beta1) + 3 * _a((1 - beta1) * gx) + _a(mi))
        vi = xf(nu) * beta2 + (1 - beta2) * gx * gx
        ev = U * (2 * _a(xf(nu) * beta2) + 4 * _a((1 - beta2) * gx * gx) + _a(vi))
    vpn, vpe, v, ve, dd, de = _step_out(vp, mi, em, vi, ev, lr, jitter)
    return vpn, vpe, mi, C * em, v, ve, dd, de


def _step_out(vp, num, enum, v, ev, lr, jitter):
    s = v + jitter
    rs = pr._sqrt(s)
    dd = num / rs
    sa = _a(s)
    edd = enum / _a(rs) + _a(dd) * (0.5 * (ev + U * sa) / sa + 2 * U)
    vpn = xf(vp) - lr * dd
    evp = lr * edd + U * (_a(lr * dd) * 2 + _a(vpn))
    return vpn, C * evp, v, C * ev, dd, C * edd


# ---- vb_dis_bisection_f64 ----------------------------------------------------------------------------------------
def dis_weights(lp, lpp, lq, eps):
    """w = exp(eps lp + (1 - eps) lpp - lq) at a float64 eps; (w, w bound, sum w, its bound, ESS, its bound)"""
    S = lq.size
    a1, a2 = xf(eps) * xf(lp), (1 - xf(eps)) * xf(lpp)
    lw = a1 + a2 - xf(lq)
    dl = U * (_a(a1) + 3 * _a(a2) + _a(a1 + a2) + _a(lw))
    v = _exp(lw)
    va = _a(v)
    rv = dl + 2 * U
    n = -(-S // 1024) + 10
    a = v.sum()
    b = (v * v).sum()
    ea = U * n * float(va.sum()) + float((va * rv).sum())
    eb = U * n * float((va * va).sum()) + float((va * va * (2 * rv + U)).sum())
    ess = a * a / b
    fa, fb = float(a), float(b)
    ress = (2 * ea / fa + eb / fb + 2 * U) if fa > 0 else np.inf
    return v, C * (va * rv + Q), a, C * ea, ess, C * ress * abs(float(ess))


def dis_bisection(lp, lpp, lq, eps_guess, max_eps, ess_target, max_its):
    """the reference's bisection with the device's float64 midpoints; per round (lower, upper, eps, ESS, bound)"""
    lower, upper = 0.0, float(eps_guess)
    eps = (lower + upper) / 2.0
    rounds = []
    for it in range(max_its + 1):
        v, _, a, _, ess, eb = dis_weights(lp, lpp, lq, eps)
        rounds.append({'lower': lower, 'upper': upper, 'eps': eps, 'ess': ess, 'bound': eb,
                       'margin': abs(float(ess - ess_target)) / eb if eb > 0 else np.inf})
        if it == max_its:
            break
        if float(ess) > ess_target:
            upper = eps
        else:
            lower = eps
        eps = (lower + upper) / 2.0
    mid = eps
    if lower == 0.0:
        eps = 0.0
    if upper == max_eps:
        eps = max_eps
    decided = rounds[:-1]
    amb = [r for r in decided if not r['margin'] > 1.0]
    return {'eps': eps, 'mid': mid, 'rounds': rounds, 'determined': not amb,
            'interval': (amb[0]['lower'], amb[0]['upper']) if amb else (eps, eps)}


# ---- cases shared by the CPU and GPU tests ----------------------------------------------------------------------
DIMS = (1, 31, 32, 33, 63, 64, 65, 257, 2048)
COUNTS = (1, 7, 8, 9, 1023, 1024, 1025)
SHAPES = [(1, 1), (31, 7), (32, 8), (33, 9), (63, 1023), (64, 1024), (65, 1025), (257, 9), (2048, 1025), (2048, 7),
          (1, 1025), (33, 1024), (257, 1023), (32, 9), (65, 8), (31, 1)]
FAMILIES = (('gauss', GAUSS, 0.0), ('t2.5', STUDENT, 2.5), ('t40', STUDENT, 40.0))
ALPHAS = (0.5, 2.0, 10.0)
LW_SPREAD = 850.0                        # nats between the largest and the smallest log-weight


def case_params(i):
    """(d, S, family name, family id, df, alpha, prior_sd) of shape i: families, alphas and the flat prior rotate"""
    d, S = SHAPES[i]
    name, fam, df = FAMILIES[i % 3]
    return d, S, name, fam, df, ALPHAS[(i // 3) % 3], (np.inf if i % 4 == 3 else 3.0)


def make_case(i):
    """host-built inputs of every entry point at shape i, float64: var_param, base draws e, theta = fl(mu + sigma e),
    ll spread over LW_SPREAD nats with its maximum at the last sample, per-sample gradients G, the alpha weights w
    (from the reference's log-weights), weights wr of the same shape (zeros included) scaled per sample for the
    gradient reduction, and a score batch (pool x, idx, weights, scale)"""
    d, S, name, fam, df, alpha, prior_sd = case_params(i)
    rs = np.random.RandomState(1000 + i)
    vp = np.concatenate([0.3 * rs.randn(d), 0.2 * rs.randn(d) - 0.3])
    e = rs.randn(S, d) if fam == GAUSS else rs.standard_t(df, size=(S, d))
    theta = to64(sample(vp, e)[0])
    ll = -LW_SPREAD * rs.rand(S) + 0.1 * rs.randn(S)
    ll[-1] = 300.0
    G = rs.randn(S, d) * np.exp(0.5 * rs.randn(d))
    lw = to64(log_weights(vp, theta, e, ll, fam, df, prior_sd)[0])
    assert np.argmax(lw) == S - 1
    w = to64(alpha_weights(lw, alpha)[0])
    pool = to64(sample(vp, rs.randn(S + 7, d) if fam == GAUSS else rs.standard_t(df, size=(S + 7, d)))[0])
    idx = rs.randint(0, S + 7, size=S).astype(np.int64)
    idx[0] = S + 6
    return dict(i=i, d=d, S=S, name=name, fam=fam, df=df, alpha=alpha, prior_sd=prior_sd, vp=vp, e=e, theta=theta,
                ll=ll, G=G, lw=lw, w=w, wr=w * (0.25 + rs.rand(S)), pool=pool, idx=idx, sw=0.5 + rs.rand(S + 7), scale=1.0 / S,
                loc=0.5 * rs.randn(d), tscale=np.exp(0.3 * rs.randn(d)), tkind=i % 2, tdf=df if df else 5.0)


def gsums(c, weighted):
    """gmu, ge (float64) the finish kernel receives: the reference reduction of G, weighted by w for ALPHA"""
    gm, _, ge, _ = reduce_grads(c['G'], c['w'] if weighted else None, c['e'])
    return to64(gm), to64(ge)
