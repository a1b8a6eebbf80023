"""The unfused mean-field kernels element by element, through the C ABI, on host-built inputs: vb_mf_sample_f64,
vb_mf_log_density_f64, vb_target_logp_grad_f64, vb_mf_reduce_grads_f64, vb_mf_alpha_weights_f64,
vb_mf_objective_finish_f64 (all three objectives), vb_mf_score_f64, the optimiser steps and the DIS bisection, each
output under its worst-case bound (tests/_mf_kernels_ref.py) at d around the 32-column blocks, S around the 8-sample
blocks and the 1024-thread blocks, and counts one past every grid-stride wrap.  Every call writes into NaN-filled
outputs followed by sentinels and is repeated three times bitwise; w = NULL must equal explicit ones and logp = NULL
must leave value and gradient unchanged, bitwise.  End to end: ExclusiveKL (both forms), AlphaDivergence and DIS
through the public API against the oracle."""
import math

import numpy as np
import pytest
import torch

import _mf_kernels_ref as R
from conftest import relerr

pytestmark = pytest.mark.gpu
SENT = -7.25e77
PAD = 8
TOL64 = 1e-10


def _L():
    from viabel_b200 import _lib
    return _lib


def _sms():
    return _L().lib.vb_device_sm_count()


def _dev(a, dtype=torch.float64):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device='cuda')


class _Pinned(list):
    """Device copies of host arrays for one C ABI call.  The copies are held here until the call has returned and
    been synchronised: a temporary passed as L.ptr(_dev(a)) is freed as soon as ptr() returns, and the caching
    allocator may then hand its block to the next argument's copy, so two arguments would alias."""

    def __call__(self, a, dtype=torch.float64):
        if a is None:
            return None
        t = _dev(a, dtype)
        self.append(t)
        return _L().ptr(t)


def _out(n):
    """n NaNs followed by PAD sentinels"""
    t = torch.full((n + PAD,), SENT, dtype=torch.float64, device='cuda')
    t[:n] = float('nan')
    return t


def _get(t, n, what):
    torch.cuda.synchronize()
    a = t.cpu().numpy()
    assert np.all(a[n:] == SENT), what + ': written past its end'
    return a[:n]


def _ws(nbytes):
    ws = torch.empty(max(int(nbytes), 8), dtype=torch.uint8, device='cuda')
    ws.fill_(0xFF)                            # NaN doubles
    return ws


def _repeat(fn):
    """fn() three times; every output bitwise equal"""
    first = fn()
    for _ in range(2):
        again = fn()
        for a, b in zip(first, again):
            assert np.array_equal(a, b, equal_nan=True), 'not bitwise reproducible'
    return first


class Ratios(dict):
    def add(self, key, dev, ref, bound):
        self[key] = max(self.get(key, 0.0), R.ratio(dev, ref, bound))

    def check(self, tag):
        print('%s: %s' % (tag, ', '.join('%s %.3g' % kv for kv in sorted(self.items()))))
        bad = {k: v for k, v in self.items() if not v <= 1.0}
        assert not bad, (tag, bad)


# ---- C ABI calls ------------------------------------------------------------------------------------------------
def call_sample(vp, e):
    L, dv = _L(), _Pinned()
    S, d = e.shape
    th = _out(S * d)
    assert L.lib.vb_mf_sample_f64(dv(vp), dv(e), L.ptr(th), S, d, L.stream()) == 0, L.last_error()
    return (_get(th, S * d, 'theta').reshape(S, d),)


def call_log_density(vp, x, fam, df):
    L, dv = _L(), _Pinned()
    n, d = x.shape
    out = _out(n)
    assert L.lib.vb_mf_log_density_f64(dv(vp), dv(x), n, d, fam, df, L.ptr(out), L.stream()) == 0
    return (_get(out, n, 'log density'),)


def call_target(theta, kind, loc, scale, df, cst, want_grad=True):
    L, dv = _L(), _Pinned()
    S, d = theta.shape
    lp, g = _out(S), _out(S * d)
    assert L.lib.vb_target_logp_grad_f64(dv(theta), S, d, kind, dv(loc), dv(scale), df, cst,
                                         L.ptr(lp), L.ptr(g) if want_grad else None, L.stream()) == 0, L.last_error()
    gg = _get(g, S * d, 'target grad')
    if not want_grad:
        assert np.all(np.isnan(gg)), 'gradient written without being asked for'
    return _get(lp, S, 'target logp'), gg.reshape(S, d)


def call_reduce(G, w, e):
    L, dv = _L(), _Pinned()
    S, d = G.shape
    gm, ge = _out(d), _out(d)
    assert L.lib.vb_mf_reduce_grads_f64(dv(G), dv(w), dv(e), S, d, L.ptr(gm), L.ptr(ge),
                                        L.stream()) == 0, L.last_error()
    return _get(gm, d, 'gmu'), _get(ge, d, 'ge')


def call_alpha(vp, theta, e, ll, fam, df, prior_sd, alpha):
    L, dv = _L(), _Pinned()
    S, d = theta.shape
    lw, w, v = _out(S), _out(S), _out(1)
    assert L.lib.vb_mf_alpha_weights_f64(dv(vp), dv(theta), dv(e), dv(ll), S, d,
                                         fam, df, prior_sd, alpha, L.ptr(lw), L.ptr(w), L.ptr(v), L.stream()) == 0, \
        L.last_error()
    return _get(lw, S, 'lw'), _get(w, S, 'w'), _get(v, 1, 'alpha value')


def call_finish(c, objective, gmu, ge, w=None, want_logp=True, want_value=True, ws_bytes=None):
    """(rc, value, grad, logp); on ALPHA the value output stays NaN (it comes from vb_mf_alpha_weights_f64)"""
    L, dv = _L(), _Pinned()
    S, d = c['theta'].shape
    v, g, lp = _out(1), _out(2 * d), _out(S)
    nb = L.lib.vb_mf_objective_finish_workspace_bytes(S) if ws_bytes is None else ws_bytes
    ws = _ws(nb)
    rc = L.lib.vb_mf_objective_finish_f64(
        dv(c['vp']), dv(c['theta']), dv(c['e']), dv(c['ll']), dv(gmu),
        dv(ge), dv(w), S, d, c['fam'], c['df'], c['prior_sd'], objective,
        c['alpha'], L.ptr(v) if want_value else None, L.ptr(g), L.ptr(lp) if want_logp else None, L.ptr(ws), nb,
        L.stream())
    vv, gg, ll = _get(v, 1, 'value'), _get(g, 2 * d, 'grad'), _get(lp, S, 'logp')
    if rc != 0:
        assert np.all(np.isnan(vv)) and np.all(np.isnan(gg)) and np.all(np.isnan(ll)), 'outputs written by a failing call'
    if not want_logp:
        assert np.all(np.isnan(ll))
    return rc, vv, gg, ll


def call_score(c, with_idx, w):
    L, dv = _L(), _Pinned()
    d = c['d']
    x = c['pool']
    n = c['S'] if with_idx else x.shape[0]
    v, g = _out(1), _out(2 * d)
    ws = _ws(L.lib.vb_mf_score_workspace_bytes(d))
    idx = dv(c['idx'], torch.int64) if with_idx else None
    assert L.lib.vb_mf_score_f64(dv(c['vp']), dv(x), idx, dv(w), c['scale'], n, d,
                                 c['fam'], c['df'], L.ptr(v), L.ptr(g), L.ptr(ws), ws.numel(), L.stream()) == 0, \
        L.last_error()
    return _get(v, 1, 'score value'), _get(g, 2 * d, 'score grad')


# ---- every entry point at each case shape --------------------------------------------------------------------------
def run_case(i):
    c = R.make_case(i)
    d, S, fam, df, alpha, psd = c['d'], c['S'], c['fam'], c['df'], c['alpha'], c['prior_sd']
    vp, e, theta = c['vp'], c['e'], c['theta']
    r = Ratios()

    (th,) = _repeat(lambda: call_sample(vp, e))
    r.add('sample', th, *R.sample(vp, e))

    (ld,) = _repeat(lambda: call_log_density(vp, theta, fam, df))
    r.add('log_density', ld, *R.log_density(vp, theta, fam, df))

    cst = -1.25 * d
    lp, tg = _repeat(lambda: call_target(theta, c['tkind'], c['loc'], c['tscale'], c['tdf'], cst))
    rlp, blp, rg, bg = R.target_logp_grad(theta, c['tkind'], c['loc'], c['tscale'], c['tdf'], cst)
    r.add('target_logp', lp, rlp, blp)
    r.add('target_grad', tg, rg, bg)
    assert np.array_equal(call_target(theta, c['tkind'], c['loc'], c['tscale'], c['tdf'], cst, False)[0], lp)

    for tag, w in (('', None), ('/w', c['wr'])):
        gm, ge = _repeat(lambda: call_reduce(c['G'], w, e))
        rgm, bgm, rge, bge = R.reduce_grads(c['G'], w, e)
        r.add('reduce_gmu' + tag, gm, rgm, bgm)
        r.add('reduce_ge' + tag, ge, rge, bge)
        if w is None:
            g1 = call_reduce(c['G'], np.ones(S), e)
            assert np.array_equal(g1[0], gm) and np.array_equal(g1[1], ge), 'w = ones differs from w = NULL'

    lw, w, av = _repeat(lambda: call_alpha(vp, theta, e, c['ll'], fam, df, psd, alpha))
    r.add('alpha_lw', lw, *R.log_weights(vp, theta, e, c['ll'], fam, df, psd))
    rw, bw, rv, bv = R.alpha_weights(lw, alpha)
    r.add('alpha_w', w, rw, bw)
    r.add('alpha_value', av, rv, bv)
    if S > 1000 and alpha > 1:
        assert np.any(w == 0.0), 'the log-weight spread should underflow some weights'

    for obj, oname in ((R.EKL, 'ekl'), (R.EKL_PATH, 'path'), (R.ALPHA, 'alpha')):
        wt = c['w'] if obj == R.ALPHA else None
        gmu, ge = R.gsums(c, obj == R.ALPHA)
        rc, v, g, lpo = _repeat(lambda: call_finish(c, obj, gmu, ge, w=wt))
        assert rc == 0, _L().last_error()
        rg, bg = R.grad(vp, theta, e, gmu, ge, c['w'], fam, df, psd, obj, alpha)
        r.add(oname + '_grad', g, rg, bg)
        if obj != R.ALPHA:
            rv, bv, rf, bf = R.value_and_logp(vp, theta, e, c['ll'], fam, df, psd, obj)
            r.add(oname + '_value', v, rv, bv)
            r.add(oname + '_logp', lpo, rf, bf)
        else:
            assert np.all(np.isnan(v)), 'AlphaDivergence value written by the finish step'
            rf, bf = R.value_and_logp(vp, theta, e, c['ll'], fam, df, psd, R.EKL)[2:]
            r.add('alpha_logp', lpo, rf, bf)
        rc2, v2, g2, _ = call_finish(c, obj, gmu, ge, w=wt, want_logp=False)
        assert rc2 == 0 and np.array_equal(v2, v, equal_nan=True) and np.array_equal(g2, g), 'logp changes the result'

    for tag, with_idx, w in (('idx', True, None), ('w', False, c['sw'])):
        v, g = _repeat(lambda: call_score(c, with_idx, w))
        rv, bv, rg, bg = R.score(vp, c['pool'], c['idx'] if with_idx else None, w, c['scale'], fam, df)
        r.add('score_value/' + tag, v, rv, bv)
        r.add('score_grad/' + tag, g, rg, bg)
    v1, g1 = call_score(c, True, np.ones(S))
    v0, g0 = call_score(c, True, None)
    assert np.array_equal(v1, v0) and np.array_equal(g1, g0), 'score: w = ones differs from w = NULL'
    return r


@pytest.mark.parametrize('i', range(len(R.SHAPES)), ids=['d%d_S%d' % s for s in R.SHAPES])
def test_kernels_elementwise(i):
    run_case(i).check(R.case_params(i))


def test_grid_stride_wraps():
    """one count past each capped grid: sample (16 SMs x 256 elements), log density and log-weights (16 SMs x 8 rows),
    the target plugin (8 SMs x 8 rows); the finish step's value at the same S (over 256 block shares)"""
    sms = _sms()
    rs = np.random.RandomState(77)
    r = Ratios()
    n_el = 16 * sms * 256 + 1
    for d in (1, 33):
        S = -(-n_el // d)
        vp = np.concatenate([rs.randn(d), 0.3 * rs.randn(d)])
        e = rs.randn(S, d)
        (th,) = _repeat(lambda: call_sample(vp, e))
        r.add('sample/d%d' % d, th, *R.sample(vp, e))
    n_rows = 16 * sms * 8 + 1
    for d, fam, df in ((3, R.GAUSS, 0.0), (2, R.STUDENT, 2.5)):
        vp = np.concatenate([rs.randn(d), 0.3 * rs.randn(d)])
        x = rs.randn(n_rows, d) * 2
        (ld,) = _repeat(lambda: call_log_density(vp, x, fam, df))
        r.add('log_density/d%d' % d, ld, *R.log_density(vp, x, fam, df))
        e = rs.randn(n_rows, d) if fam == R.GAUSS else rs.standard_t(df, size=(n_rows, d))
        theta = R.to64(R.sample(vp, e)[0])
        ll = -R.LW_SPREAD * rs.rand(n_rows)
        lw, w, av = _repeat(lambda: call_alpha(vp, theta, e, ll, fam, df, 3.0, 2.0))
        r.add('alpha_lw/d%d' % d, lw, *R.log_weights(vp, theta, e, ll, fam, df, 3.0))
        rw, bw, rv, bv = R.alpha_weights(lw, 2.0)
        r.add('alpha_w/d%d' % d, w, rw, bw)
        r.add('alpha_value/d%d' % d, av, rv, bv)
        c = dict(vp=vp, theta=theta, e=e, ll=ll, fam=fam, df=df, prior_sd=3.0, alpha=2.0, d=d, S=n_rows)
        gmu, ge = np.zeros(d), np.zeros(d)
        for obj in (R.EKL, R.EKL_PATH):
            rc, v, g, lp = _repeat(lambda: call_finish(c, obj, gmu, ge))
            assert rc == 0
            rv, bv, rf, bf = R.value_and_logp(vp, theta, e, ll, fam, df, 3.0, obj)
            r.add('finish_value/d%d/%d' % (d, obj), v, rv, bv)
            r.add('finish_logp/d%d/%d' % (d, obj), lp, rf, bf)
    S = 8 * sms * 8 + 1
    for kind, df in ((0, 0.0), (1, 3.0)):
        theta = rs.randn(S, 5) * 3
        loc, sc = rs.randn(5), np.exp(rs.randn(5) * 0.3)
        lp, g = _repeat(lambda: call_target(theta, kind, loc, sc, df, 0.5))
        rlp, blp, rg, bg = R.target_logp_grad(theta, kind, loc, sc, df, 0.5)
        r.add('target_logp/%d' % kind, lp, rlp, blp)
        r.add('target_grad/%d' % kind, g, rg, bg)
    r.check('wraps')


# ---- optimiser steps -------------------------------------------------------------------------------------------
def _opt_call(kind, vp, g, m, nu, first, want_dir, lr=0.05):
    L = _L()
    P = vp.size
    bufs = {}
    for k, a in (('vp', vp), ('m', m), ('nu', nu)):
        t = torch.full((P + PAD,), SENT, dtype=torch.float64, device='cuda')
        t[:P] = _dev(a)
        bufs[k] = t
    dr = _out(P)
    gd = _dev(g)
    if kind == 'rmsprop':
        rc = L.lib.vb_rmsprop_step_f64(L.ptr(bufs['vp']), L.ptr(gd), L.ptr(bufs['nu']), L.ptr(dr) if want_dir else None,
                                       P, lr, 0.9, 1e-8, int(first), L.stream())
    else:
        rc = L.lib.vb_adam_step_f64(L.ptr(bufs['vp']), L.ptr(gd), L.ptr(bufs['m']), L.ptr(bufs['nu']),
                                    L.ptr(dr) if want_dir else None, P, lr, 0.9, 0.999, 1e-8, int(first), L.stream())
    assert rc == 0, L.last_error()
    out = [_get(bufs[k], P, k) for k in ('vp', 'm', 'nu')] + [_get(dr, P, 'direction')]
    if not want_dir:
        assert np.all(np.isnan(out[3]))
    return out


@pytest.mark.parametrize('P', [1, 1000, 1_000_003])
@pytest.mark.parametrize('kind', ['rmsprop', 'adam'])
def test_optimizer_steps(kind, P):
    """one past the 8 SMs x 256 grid at P = 1 000 003 (sms permitting); the first and a later step; gradients from
    1e-12 to 1e6 and zeros"""
    rs = np.random.RandomState(P)
    vp = rs.randn(P)
    g = rs.randn(P) * np.exp(rs.uniform(-28, 14, P))
    g[::97] = 0.0
    m, nu = rs.randn(P) * 0.1, rs.rand(P) * 0.01
    r = Ratios()
    for first in (1, 0):
        vpo, mo, nuo, dro = _repeat(lambda: _opt_call(kind, vp, g, m, nu, first, True))
        nd = _opt_call(kind, vp, g, m, nu, first, False)
        assert np.array_equal(nd[0], vpo) and np.array_equal(nd[2], nuo), 'direction = NULL changes the step'
        if kind == 'rmsprop':
            rvp, bvp, rnu, bnu, rdd, bdd = R.rmsprop(vp, g, nu, 0.05, 0.9, 1e-8, first)
            assert np.array_equal(mo, m), 'RMSProp wrote m'
        else:
            rvp, bvp, rm, bm, rnu, bnu, rdd, bdd = R.adam(vp, g, m, nu, 0.05, 0.9, 0.999, 1e-8, first)
            r.add('m/%d' % first, mo, rm, bm)
        r.add('vp/%d' % first, vpo, rvp, bvp)
        r.add('nu/%d' % first, nuo, rnu, bnu)
        r.add('dir/%d' % first, dro, rdd, bdd)
    r.check((kind, P))


# ---- DIS ---------------------------------------------------------------------------------------------------------
def _dis_call(lp, lpp, lq, eps_guess, target, max_its=50):
    L, dv = _L(), _Pinned()
    S = lq.size
    w, out = _out(S), _out(4)
    assert L.lib.vb_dis_bisection_f64(dv(lp), dv(lpp), dv(lq), S, eps_guess, 1.0, target,
                                      max_its, L.ptr(w), L.ptr(out), L.stream()) == 0, L.last_error()
    return _get(w, S, 'dis w'), _get(out, 4, 'dis out')


def check_bisection(lp, lpp, lq, eps_guess, target, r, tag):
    ref = R.dis_bisection(lp, lpp, lq, eps_guess, 1.0, target, 50)
    w, out = _repeat(lambda: _dis_call(lp, lpp, lq, eps_guess, target))
    eps = out[0]
    if ref['determined']:
        assert eps == ref['eps'], (tag, eps, ref['eps'])
        mid = ref['mid']
    else:
        lo, hi = ref['interval']
        assert lo <= eps <= hi, (tag, eps, lo, hi)
        mid = eps if 0.0 < eps < 1.0 else None
    assert out[2] == 0.0
    if mid is not None:
        v, bv, a, ba, ess, be = R.dis_weights(lp, lpp, lq, mid)
        r.add('dis_w/' + tag, w, v, bv)
        r.add('dis_sw/' + tag, out[3], a, ba)
        r.add('dis_ess/' + tag, out[1], ess, be)
    return ref, eps


def _dis_vectors(S, d, seed, tight):
    rs = np.random.RandomState(seed)
    x = rs.randn(S, d) * 1.5
    lq = -0.5 * np.sum((x / 1.5) ** 2, axis=1) - d * np.log(1.5 * np.sqrt(2 * np.pi))
    lpp = -0.5 * np.sum((x / tight) ** 2, axis=1)
    lp = -0.5 * np.sum(x ** 2, axis=1)
    return lp, lpp, lq


@pytest.mark.parametrize('S', [1, 7, 1023, 1024, 1025, 5000])
def test_dis_bisection(S):
    """the tempering search at counts around the one 1024-thread block; interior, eps = 0 and eps = 1 ends; a guess
    below one; the ESS margin of every round against its bound decides bit-equality"""
    r = Ratios()
    determined = 0
    for j, (tight, frac, guess) in enumerate(((0.6, 0.3, 1.0), (1.4, 0.15, 1.0), (0.2, 0.999, 1.0), (0.6, 0.3, 0.37))):
        lp, lpp, lq = _dis_vectors(S, 4, S + j, tight)
        ref, _ = check_bisection(lp, lpp, lq, guess, frac * S, r, '%d' % j)
        determined += ref['determined']
    print('S = %d: %d of 4 determined' % (S, determined))
    r.check(('dis', S))


@pytest.mark.parametrize('resample', [False, True])
def test_dis_objective_large(resample):
    """DISInclusiveKL at S = 5000, d = 70 through the public API: epsilon against the bisection reference, value and
    gradient against the score reference at the objective's own weights and resampled indices"""
    import viabel_b200 as vb
    S, d = 5000, 70
    rs = np.random.RandomState(5)
    mean, sd = rs.randn(d), np.exp(0.3 * rs.randn(d))
    fam = vb.MFStudentT(d, 40.0) if resample else vb.MFGaussian(d)
    prior_param = np.concatenate([np.zeros(d), np.ones(d)])
    obj = vb.DISInclusiveKL(fam, vb.GaussianTarget(mean, sd), S, 1500, vb.MFGaussian(d), prior_param,
                            use_resampling=resample)
    vp = np.concatenate([mean + 0.1 * rs.randn(d), np.log(sd) + 0.1])
    r = Ratios()
    for call in range(2):
        np.random.seed(100 + call)
        eps_in = float(obj._eps)
        value, grad = obj(vp)
        x = obj._state_samples.cpu().numpy()
        lq, lpp = obj._state_log_q.cpu().numpy(), obj._state_log_p.cpu().numpy()
        lp = vb.MFGaussian(d).log_density(_dev(prior_param), obj._state_samples).cpu().numpy()
        ref = R.dis_bisection(lp, lpp, lq, eps_in, 1.0, 1500, 50)
        lo, hi = ref['interval']
        assert (obj._eps == ref['eps']) if ref['determined'] else (lo <= obj._eps <= hi), (obj._eps, ref['interval'])
        w = obj._state_w.cpu().numpy()
        famid, df = (R.STUDENT, 40.0) if resample else (R.GAUSS, 0.0)
        if resample:
            np.random.seed(100 + call)
            p = obj._state_w_normalized.cpu().numpy()
            idx = obj._resample_indices(S, p)
            rv, bv, rg, bg = R.score(vp, x, idx, None, float(obj._state_w_sum) / S / idx.size, famid, df)
        else:
            rv, bv, rg, bg = R.score(vp, x, None, w, 1.0 / S, famid, df)
        r.add('value', value, rv, bv)
        r.add('grad', grad, rg, bg)
    r.check(('dis_large', resample))


# ---- argument errors ---------------------------------------------------------------------------------------------
def test_finish_argument_errors():
    """bad family, df <= 2, S <= 0, ALPHA without w, grad without gmu / ge, a workspace one double short: each an
    error return with nothing written"""
    L, dv = _L(), _Pinned()
    c = R.make_case(3)
    gmu, ge = R.gsums(c, False)
    good = call_finish(c, R.EKL, gmu, ge)
    assert good[0] == 0
    for kw, rc_want in ((dict(fam=7), L.VB_ERR_INVALID_ARG), (dict(fam=R.STUDENT, df=2.0), L.VB_ERR_INVALID_ARG),
                        (dict(fam=R.STUDENT, df=-1.0), L.VB_ERR_INVALID_ARG)):
        assert call_finish(dict(c, **kw), R.EKL, gmu, ge)[0] == rc_want, kw
    assert call_finish(c, R.ALPHA, gmu, ge, w=None)[0] == L.VB_ERR_INVALID_ARG
    assert call_finish(c, R.EKL, gmu, ge, ws_bytes=L.lib.vb_mf_objective_finish_workspace_bytes(c['S']) - 8)[0] \
        == L.VB_ERR_WORKSPACE
    assert call_finish(c, R.EKL, gmu, ge, want_value=False)[0] == L.VB_ERR_INVALID_ARG
    assert L.lib.vb_mf_objective_finish_workspace_bytes(0) == 0
    assert L.lib.vb_mf_objective_finish_workspace_bytes(17) == 24
    S, d = c['theta'].shape
    vp, th, e, ll = (_dev(c[k]) for k in ('vp', 'theta', 'e', 'll'))
    ws = _ws(L.lib.vb_mf_objective_finish_workspace_bytes(S))
    for S_bad in (0, -1):
        v = _out(1)
        assert L.lib.vb_mf_objective_finish_f64(L.ptr(vp), L.ptr(th), L.ptr(e), L.ptr(ll), None, None, None, S_bad, d,
                                                0, 0.0, 3.0, R.EKL, 0.0, L.ptr(v), None, None, L.ptr(ws), ws.numel(),
                                                L.stream()) == L.VB_ERR_INVALID_ARG
        assert np.isnan(_get(v, 1, 'value')[0])
    g = _out(2 * d)
    assert L.lib.vb_mf_objective_finish_f64(L.ptr(vp), L.ptr(th), L.ptr(e), L.ptr(ll), None, dv(ge), None, S,
                                            d, 0, 0.0, 3.0, R.EKL, 0.0, None, L.ptr(g), None, L.ptr(ws), ws.numel(),
                                            L.stream()) == L.VB_ERR_INVALID_ARG
    assert np.all(np.isnan(_get(g, 2 * d, 'grad')))
    # gradient only: no value, no logp, no workspace
    assert L.lib.vb_mf_objective_finish_f64(L.ptr(vp), L.ptr(th), L.ptr(e), L.ptr(ll), dv(gmu), dv(ge),
                                            None, S, d, 0, 0.0, c['prior_sd'], R.EKL, 0.0, None, L.ptr(g), None, None, 0,
                                            L.stream()) == 0
    assert np.array_equal(_get(g, 2 * d, 'grad'), good[2])


# ---- end to end through the public API -------------------------------------------------------------------------
def _hier_shape(d):
    """(G, p) with d = (G + 1) p + 2 and at most 32 coefficients per group (the plugin's limit)"""
    return {33: (30, 1), 257: (14, 17), 2048: (65, 31)}[d]


def _models(vb, vo, name, d):
    rs = np.random.RandomState(d)
    if name == 'gauss':
        mean, sd = rs.randn(d), np.exp(0.5 * rs.randn(d))
        return vb.GaussianTarget(mean, sd), lambda th: vo.gauss_target_logp_grad(th, mean, sd)
    if name == 'student':
        loc, sc = rs.randn(d), np.exp(0.5 * rs.randn(d))
        return vb.StudentTTarget(loc, sc, 4.0), lambda th: vo.student_target_logp_grad(th, loc, sc, 4.0)
    if name == 'hier':
        G, p = _hier_shape(d)
        n_per = 4
        N = G * n_per
        group = np.repeat(np.arange(G), n_per)
        X = rs.randn(N, p)
        y = X @ rs.randn(p) + 0.3 * rs.randn(N)
        return (vb.HierarchicalLinearRegression(X, y, group, G),
                lambda th: vo.hier_linear_logp_grad(th, X, y, group, G, p))
    loc, sc = rs.randn(d), np.exp(0.5 * rs.randn(d))
    lt, st = _dev(loc), _dev(sc)
    c = math.lgamma(3.5) - math.lgamma(3.0) - 0.5 * math.log(6.0 * math.pi)

    def logp(x):
        z = (x - lt) / st
        return (c - 3.5 * torch.log1p(z * z / 6.0) - torch.log(st)).sum(dim=1)
    return vb.Model(logp), lambda th: vo.student_target_logp_grad(th, loc, sc, 6.0)


@pytest.mark.parametrize('S', [9, 1025])
@pytest.mark.parametrize('d', [33, 257, 2048])
@pytest.mark.parametrize('model', ['gauss', 'student', 'hier', 'user'])
def test_objectives_end_to_end(model, d, S):
    import viabel_b200 as vb
    from oracle import viabel_oracle as vo
    m, om = _models(vb, vo, model, d)
    student = (d + S) % 2 == 0
    fam = vb.MFStudentT(d, 5.0) if student else vb.MFGaussian(d)
    kw = dict(family='t', df=5.0) if student else dict(family='gaussian')
    rs = np.random.RandomState(S + d)
    vp = np.concatenate([0.2 * rs.randn(d), -0.5 + 0.1 * rs.randn(d)])
    base = rs.standard_t(5.0, size=(S, d)) if student else rs.randn(S, d)
    for path in (False, True):
        v, g = vb.ExclusiveKL(fam, m, S, use_path_deriv=path)(vp, base=base)
        v0, g0, _ = vo.exclusive_kl_meanfield(vp, base, om, path_deriv=path, **kw)
        assert relerr(v, v0) < TOL64 and relerr(g, g0) < TOL64, (path, relerr(v, v0), relerr(g, g0))
        v2, g2 = vb.ExclusiveKL(fam, m, S, use_path_deriv=path)(vp, base=base)
        assert v2 == v and np.array_equal(g2, g), 'ExclusiveKL not bitwise reproducible'
    for alpha in (0.5, 2.0):
        v, g = vb.AlphaDivergence(fam, m, S, alpha)(vp, base=base)
        v0, g0, _ = vo.alpha_divergence_meanfield(vp, base, om, alpha, **kw)
        assert relerr(v, v0) < TOL64 and relerr(g, g0) < TOL64, (alpha, relerr(v, v0), relerr(g, g0))
