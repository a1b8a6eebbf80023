"""CPU: the reference of the unfused mean-field kernels (tests/_mf_kernels_ref.py) against torch autograd of its own
expressions, and its bounds against mutated kernels -- each mutation must put some output element outside its bound
at every case shape of tests/test_gpu_mf_kernels.py it applies to."""
import functools
import math

import numpy as np
import pytest
import torch

import _mf_kernels_ref as R
from _philox_ref import to64

FAMS = [('gauss', R.GAUSS, 0.0), ('t2.5', R.STUDENT, 2.5), ('t40', R.STUDENT, 40.0)]


def _t(a):
    return torch.as_tensor(np.asarray(a, dtype=np.float64))


def _lq_torch(x, mu, ls, fam, df):
    z = (x - mu) / torch.exp(ls)
    if fam == R.GAUSS:
        t = -0.5 * z * z - 0.5 * math.log(2 * math.pi)
    else:
        c = math.lgamma(0.5 * (df + 1)) - math.lgamma(0.5 * df) - 0.5 * math.log(df * math.pi)
        t = c - 0.5 * (df + 1) * torch.log1p(z * z / df)
    return (t - ls).sum(dim=1)


def _problem(fam, df, d=5, S=11, seed=3, flat_model=False):
    rs = np.random.RandomState(seed)
    vp = np.concatenate([0.3 * rs.randn(d), 0.2 * rs.randn(d) - 0.3])
    e = rs.randn(S, d) if fam == R.GAUSS else rs.standard_t(df, size=(S, d))
    loc, sc = rs.randn(d), np.exp(0.3 * rs.randn(d))
    if flat_model:
        f = lambda th: 0.0 * th.sum(dim=1) + 1.5
    else:
        f = lambda th: (-0.5 * ((th - _t(loc)) / _t(sc)) ** 2).sum(dim=1)
    theta = to64(R.sample(vp, e)[0])
    ll = f(_t(theta)).numpy()
    G = np.zeros((S, d)) if flat_model else -(theta - loc) / sc ** 2
    return vp, e, theta, ll, G, f


@pytest.mark.parametrize('fam,df', [(f, df) for _, f, df in FAMS], ids=[n for n, _, _ in FAMS])
@pytest.mark.parametrize('objective', [R.EKL, R.EKL_PATH, R.ALPHA], ids=['ekl', 'path', 'alpha'])
@pytest.mark.parametrize('prior_sd', [3.0, np.inf])
def test_reference_matches_autograd(fam, df, objective, prior_sd):
    """value and gradient wrt [mu, log sigma] of the reference's finish step (reduce_grads -> grad) against torch
    autograd through theta = mu + sigma e of the same expression"""
    d, S, alpha = 5, 11, 2.0
    vp, e, theta, ll, G, f = _problem(fam, df)
    lam = _t(vp).requires_grad_(True)
    mu, ls = lam[:d], lam[d:]
    th = mu + torch.exp(ls) * _t(e)
    if np.isfinite(prior_sd):
        prior = -0.5 * (th * th).sum(dim=1) / prior_sd ** 2 - d * math.log(prior_sd * math.sqrt(2 * math.pi))
    else:
        prior = 0.0 * th.sum(dim=1)
    lp = f(th) + prior
    w = None
    if objective == R.EKL:
        H = ls.sum() + (0.5 * d * (1 + math.log(2 * math.pi)) if fam == R.GAUSS else 0.0)
        value = -(lp.mean() + H)
        (g_t,) = torch.autograd.grad(value, lam)
    elif objective == R.EKL_PATH:
        value = -(lp - _lq_torch(th, mu.detach(), ls.detach(), fam, df)).mean()
        (g_t,) = torch.autograd.grad(value, lam)
    else:
        lw_t = lp - _lq_torch(th, mu, ls, fam, df)
        m = lw_t.max().detach()
        sv = torch.exp(lw_t - m) ** alpha
        value = torch.log(sv.mean()) / alpha + m
        (g_t,) = torch.autograd.grad(alpha * (sv.detach() * lw_t).mean(), lam)
        lw = to64(R.log_weights(vp, theta, e, ll, fam, df, prior_sd)[0])
        np.testing.assert_allclose(lw, lw_t.detach().numpy(), rtol=1e-12, atol=1e-12)
        w = to64(R.alpha_weights(lw, alpha)[0])
    gm, _, ge, _ = R.reduce_grads(G, w, e)
    g_ref = to64(R.grad(vp, theta, e, to64(gm), to64(ge), w, fam, df, prior_sd, objective, alpha)[0])
    if objective == R.ALPHA:
        v_ref = to64(R.alpha_weights(lw, alpha)[2])
    else:
        v_ref = to64(R.value_and_logp(vp, theta, e, ll, fam, df, prior_sd, objective)[0])
    np.testing.assert_allclose(v_ref, float(value.detach()), rtol=1e-12)
    np.testing.assert_allclose(g_ref, g_t.numpy(), rtol=1e-11, atol=1e-12 * np.abs(g_t.numpy()).max())


@pytest.mark.parametrize('fam,df', [(f, df) for _, f, df in FAMS], ids=[n for n, _, _ in FAMS])
def test_alpha_sw_term(fam, df):
    """with a constant model and a flat prior the AlphaDivergence gradient wrt log sigma is alpha / S sum_s w_s, the
    sw term alone (d(-log q(theta(lambda); lambda)) / d log sigma_j = 1), and zero wrt mu"""
    d, S, alpha = 5, 11, 0.5
    vp, e, theta, ll, G, f = _problem(fam, df, flat_model=True)
    lw = to64(R.log_weights(vp, theta, e, ll, fam, df, np.inf)[0])
    w = to64(R.alpha_weights(lw, alpha)[0])
    g = to64(R.grad(vp, theta, e, np.zeros(d), np.zeros(d), w, fam, df, np.inf, R.ALPHA, alpha)[0])
    assert np.all(g[:d] == 0)
    np.testing.assert_allclose(g[d:], alpha / S * w.sum(), rtol=1e-14)
    lam = _t(vp).requires_grad_(True)
    th = lam[:d] + torch.exp(lam[d:]) * _t(e)
    lw_t = f(th) - _lq_torch(th, lam[:d], lam[d:], fam, df)
    sv = torch.exp(lw_t - lw_t.max().detach()) ** alpha
    (g_t,) = torch.autograd.grad(alpha * (sv.detach() * lw_t).mean(), lam)
    np.testing.assert_allclose(g, g_t.numpy(), rtol=1e-12, atol=1e-15)


@pytest.mark.parametrize('fam,df', [(f, df) for _, f, df in FAMS], ids=[n for n, _, _ in FAMS])
def test_score_and_target_match_autograd(fam, df):
    """the score value and gradient (DIS) and the product target's gradient against autograd"""
    d, n = 6, 9
    rs = np.random.RandomState(9)
    vp = np.concatenate([rs.randn(d), 0.3 * rs.randn(d)])
    x = rs.randn(13, d) * 2
    idx = rs.randint(0, 13, size=n)
    w = rs.rand(n)
    v, _, g, _ = R.score(vp, x, idx, w, 0.3, fam, df)
    lam = _t(vp).requires_grad_(True)
    val = -(0.3 * _t(w) * _lq_torch(_t(x[idx]), lam[:d], lam[d:], fam, df)).sum()
    (g_t,) = torch.autograd.grad(val, lam)
    np.testing.assert_allclose(to64(v), float(val.detach()), rtol=1e-13)
    np.testing.assert_allclose(to64(g), g_t.numpy(), rtol=1e-12, atol=1e-14)
    loc, sc = rs.randn(d), np.exp(0.3 * rs.randn(d))
    th = _t(x).requires_grad_(True)
    for kind, tdf in ((0, 0.0), (1, 3.0)):
        z = (th - _t(loc)) / _t(sc)
        t = -0.5 * z * z if kind == 0 else -0.5 * (tdf + 1) * torch.log1p(z * z / tdf)
        (gt,) = torch.autograd.grad(t.sum(), th)
        lp, _, gr, _ = R.target_logp_grad(x, kind, loc, sc, tdf, 0.25)
        np.testing.assert_allclose(to64(lp), t.detach().sum(dim=1).numpy() + 0.25, rtol=1e-13)
        np.testing.assert_allclose(to64(gr), gt.numpy(), rtol=1e-13, atol=1e-15)


def test_dis_bisection_reference():
    """an interior epsilon is decided bit for bit for 40 rounds and then placed within 1e-11; an end point is decided in
    every round; a target equal to the first round's ESS leaves the whole interval open"""
    rs = np.random.RandomState(1025)
    x = rs.randn(1025, 4) * 1.5
    lq = -0.5 * np.sum((x / 1.5) ** 2, axis=1) - 4 * np.log(1.5 * np.sqrt(2 * np.pi))
    lp, lpp = -0.5 * np.sum(x ** 2, axis=1), -0.5 * np.sum((x / 0.6) ** 2, axis=1)
    ref = R.dis_bisection(lp, lpp, lq, 1.0, 1.0, 0.3 * 1025, 50)
    assert len(ref['rounds']) == 51 and not ref['determined']
    first = min(k for k, r in enumerate(ref['rounds'][:-1]) if not r['margin'] > 1)
    lo, hi = ref['interval']
    assert first >= 40 and lo <= ref['eps'] <= hi and hi - lo < 1e-11
    end = R.dis_bisection(lp, -0.5 * np.sum((x / 1.4) ** 2, axis=1), lq, 1.0, 1.0, 0.15 * 1025, 50)
    assert end['determined'] and end['eps'] == 0.0
    amb = R.dis_bisection(lp, lpp, lq, 1.0, 1.0, float(ref['rounds'][0]['ess']), 50)
    assert not amb['determined'] and amb['interval'] == (0.0, 1.0)


# ---- mutations ---------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def _case(i):
    return R.make_case(i)


def _fails(dev_ext, ref, bound):
    return R.ratio(to64(dev_ext), ref, bound) > 1.0


def _m_value_last_sample(c):
    acc, acc_err, _, _ = R.value_terms(c['vp'], c['theta'], c['e'], c['ll'], c['fam'], c['df'], c['prior_sd'], R.EKL)
    ref, bound = R.value_from_terms(acc, acc_err, c['vp'], c['d'], c['fam'], R.EKL)
    acc2 = acc.copy()
    acc2[-1] = 0
    return _fails(R.value_from_terms(acc2, acc_err, c['vp'], c['d'], c['fam'], R.EKL)[0], ref, bound)


def _m_last_column(c):
    gm, bgm, ge, bge = R.reduce_grads(c['G'], c['wr'], c['e'])
    g2 = gm.copy()
    g2[-1] = 0
    return _fails(g2, gm, bgm)


def _m_ge_theta(c):
    _, _, ge, bge = R.reduce_grads(c['G'], c['wr'], c['e'])
    return _fails(R.reduce_grads(c['G'], c['wr'], c['theta'])[2], ge, bge)


def _pieces(c, objective, family=None):
    w = c['w'] if objective == R.ALPHA else None
    return R.grad_pieces(c['vp'], c['theta'], c['e'], w, c['fam'] if family is None else family, c['df'], objective)


def _assemble(c, P, E, objective):
    gmu, ge = R.gsums(c, objective == R.ALPHA)
    return R.grad_assemble(P, E, c['vp'], gmu, ge, c['prior_sd'], objective, c['alpha'], c['S'])


def _m_prior_one_coord(c):
    if not np.isfinite(c['prior_sd']):
        return None
    P, E = _pieces(c, R.EKL)
    ref, bound = _assemble(c, P, E, R.EKL)
    P2 = dict(P, p1=P['p1'].copy())
    P2['p1'][-1] = 0
    return _fails(_assemble(c, P2, E, R.EKL)[0], ref, bound)


def _m_alpha_sw(c):
    P, E = _pieces(c, R.ALPHA)
    ref, bound = _assemble(c, P, E, R.ALPHA)
    return _fails(_assemble(c, dict(P, sw=0 * P['sw']), E, R.ALPHA)[0], ref, bound)


def _m_student_factor(c):
    if c['fam'] != R.STUDENT:
        return None
    P, E = _pieces(c, R.EKL_PATH)
    ref, bound = _assemble(c, P, E, R.EKL_PATH)
    Pg, _ = _pieces(c, R.EKL_PATH, family=R.GAUSS)
    return _fails(_assemble(c, dict(P, pa=Pg['pa'], pb=Pg['pb']), E, R.EKL_PATH)[0], ref, bound)


def _m_reduce_no_w(c):
    gm, bgm, ge, bge = R.reduce_grads(c['G'], c['wr'], c['e'])
    m = R.reduce_grads(c['G'], None, c['e'])
    return _fails(m[0], gm, bgm) or _fails(m[2], ge, bge)


def _m_score_no_idx(c):
    rv, bv, rg, bg = R.score(c['vp'], c['pool'], c['idx'], None, c['scale'], c['fam'], c['df'])
    mv, _, mg, _ = R.score(c['vp'], c['pool'][:c['S']], None, None, c['scale'], c['fam'], c['df'])
    return _fails(mg, rg, bg) or _fails(mv, rv, bv)


def _m_alpha_max_1024(c):
    if c['S'] <= 1024:
        return None
    rw, bw, rv, bv = R.alpha_weights(c['lw'], c['alpha'])
    return _fails(R.alpha_weights(c['lw'], c['alpha'], m=float(np.max(c['lw'][:1024])))[0], rw, bw)


MUTATIONS = {'value_drops_last_sample': _m_value_last_sample, 'reduce_drops_last_column': _m_last_column,
             'ge_uses_theta': _m_ge_theta, 'prior_dropped_on_one_coordinate': _m_prior_one_coord,
             'alpha_grad_drops_sw': _m_alpha_sw, 'path_drops_student_factor': _m_student_factor,
             'reduce_ignores_w': _m_reduce_no_w, 'score_ignores_idx': _m_score_no_idx,
             'alpha_max_over_first_1024': _m_alpha_max_1024}


@pytest.mark.parametrize('name', sorted(MUTATIONS))
def test_mutation_fails_bound(name):
    applied, missed = 0, []
    for i in range(len(R.SHAPES)):
        hit = MUTATIONS[name](_case(i))
        if hit is None:
            continue
        applied += 1
        if not hit:
            missed.append(R.SHAPES[i])
    assert applied >= 1
    assert not missed, (name, missed)


def test_reference_within_its_own_bound_after_rounding():
    """the float64 rounding of every reference output is far inside its bound (the bound is not vacuous the other way:
    the mutations above fail it)"""
    c = _case(8)
    gm, bgm, ge, bge = R.reduce_grads(c['G'], c['wr'], c['e'])
    assert R.ratio(to64(gm), gm, bgm) < 0.1 and R.ratio(to64(ge), ge, bge) < 0.1
    v, bv, f, bf = R.value_and_logp(c['vp'], c['theta'], c['e'], c['ll'], c['fam'], c['df'], c['prior_sd'], R.EKL)
    assert R.ratio(to64(v), v, bv) < 0.1 and R.ratio(to64(f), f, bf) < 0.1
