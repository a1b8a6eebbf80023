"""The batched PSIS kernel (vb_psislw_batch_f64: one CTA per column, the whole matrix in one launch) against
oracle.viabel_oracle.psislw_1d column by column: maximum and shifted cutoff bit-equal, n2 equal (so the tail set is
exact), k-hat to 1e-10 with the same +inf pattern, outputs and log-sum-exp to 1e-10.  Columns are built to reach each
rule of the one-column algorithm (tests/_psis_ref.py builds the same edges for the one-column pipeline); shapes cover
the tail-length rule, the shared-memory limit and the fallback above it, grid and 64-bit offset edges, every output
mode, bitwise repeatability, psisloo and the 2-D psislw API, and every C ABI error."""
import ctypes
import math

import numpy as np
import pytest
import torch

import _psis_ref as P
from _problems import _t_ratio, psis_case

pytestmark = pytest.mark.gpu
TOL = 1e-10
R_KHAT, R_SIGMA, R_N2, R_CUTOFF, R_LSE, R_MAX, R_STATUS, R_SUMV, R_SUMEXP2V, R_M, R_NCAND, R_SMOOTHED = range(12)
LOG_TINY = math.log(np.finfo(float).tiny)


@pytest.fixture(scope='module')
def vb():
    import viabel_b200
    return viabel_b200


@pytest.fixture(scope='module')
def psis():
    from viabel_b200 import _psis
    return _psis


@pytest.fixture(scope='module')
def vo():
    from oracle import viabel_oracle
    return viabel_oracle


def _same(a, b):
    """Bit-equal, or both NaN."""
    a, b = np.float64(a), np.float64(b)
    return a.tobytes() == b.tobytes() or (np.isnan(a) and np.isnan(b))


def _close(got, ref, what):
    if np.isfinite(ref):
        assert abs(got - ref) <= TOL * abs(ref) + 1e-300, (what, got, ref)
    else:
        assert _same(got, ref) or got == ref, (what, got, ref)


def _check_col(x, reff, row, khat, out=None, loo=None, what=''):
    """One column of a batched run against the oracle."""
    ref = P.oracle(x, reff)
    assert _same(row[R_MAX], ref['max']) and _same(row[R_CUTOFF], ref['xcut']), \
        (what, row[R_MAX], ref['max'], row[R_CUTOFF], ref['xcut'])
    assert int(row[R_N2]) == ref['n2'] and int(row[R_M]) == ref['M'], (what, row[R_N2], ref['n2'], row[R_M], ref['M'])
    assert _same(row[R_KHAT], khat), what
    if np.isfinite(ref['k']):
        _close(khat, ref['k'], (what, 'k'))
    else:
        assert khat == ref['k'], (what, khat, ref['k'])
    assert row[R_SMOOTHED] == float(ref['k'] >= 1.0 / 3.0 and np.isfinite(ref['k'])), what
    _close(row[R_LSE], ref['lse'], (what, 'lse'))
    if out is not None:
        np.testing.assert_allclose(out, ref['out'], rtol=TOL, atol=TOL, err_msg=str(what))
    if loo is not None:
        with np.errstate(all='ignore'):
            t = ref['out'] - x
            mx = np.max(t)
            ref_loo = np.log(np.sum(np.exp(t - mx))) + mx
        _close(loo, ref_loo, (what, 'loo'))
    return ref


def _run(psis, cols, reff=1.0, out=True, loo=True):
    """cols: list of 1-D arrays of equal length -> device call on the F-ordered matrix; numpy results."""
    X = np.stack(cols, axis=1)
    t = torch.from_numpy(np.ascontiguousarray(X.T)).cuda().t()
    o = torch.empty_like(t) if out else None
    o, k, r, lo = psis.psislw_batch_device(t, o, reff, want_loo=loo, want_result=True)
    return (None if o is None else o.cpu().numpy(), k.cpu().numpy(), r.cpu().numpy(),
            None if lo is None else lo.cpu().numpy())


def _check_all(psis, cols, reff=1.0, what=''):
    out, k, r, loo = _run(psis, cols, reff)
    refs = []
    for j, x in enumerate(cols):
        refs.append(_check_col(x, reff, r[j], k[j], out[:, j], loo[j], (what, j)))
    return refs


# ---- column contents ---------------------------------------------------------------------------------------------
def _rank_desc(x):
    return np.argsort(-x, kind='stable')


def _capped_pareto(n, seed):
    """k-hat above 1 whose largest smoothed values pass 0 and are clipped: log-Pareto(0.7) draws with the two largest
    lowered to the third."""
    rs = np.random.RandomState(seed)
    x = np.log(rs.pareto(0.7, n) + 1.0)
    o = np.argsort(x)
    x[o[-2:]] = x[o[-3]]
    return x


def _tie_straddle(n, reff=1.0):
    x = _t_ratio(n, 4, 9, 40)
    M = P.plan(n, reff)['M']
    r = _rank_desc(x)
    x[r[M - 6:M + 7]] = x[r[M]]                      # a tie block across rank M+1
    return x


def _signed_zeros(n):
    x = _t_ratio(n, 5, 7, 41)
    M = P.plan(n)['M']
    x -= np.sort(x)[::-1][M]                         # the (M+1)-th largest becomes 0
    r = _rank_desc(x)
    blk = r[M - 10:M + 10]
    x[blk] = np.where(np.arange(blk.size) % 2 == 0, 0.0, -0.0)
    return x


def _huge_pm(n):
    rs = np.random.RandomState(42)
    x = np.full(n, -1.5e308)
    x[rs.choice(n, 50, replace=False)] = rs.standard_t(3, 50)
    x[n // 3] = 1e308
    return x


def _floor(n):
    """Fewer than M+1 draws above log(DBL_MIN) relative to the maximum: the cutoff is the floor, n2 = 100."""
    rs = np.random.RandomState(43)
    x = -800.0 - np.abs(rs.standard_t(3, n))
    x[rs.choice(n, 100, replace=False)] = rs.standard_t(4, 100)
    return x


def _ulp_above(n):
    x = _t_ratio(n, 5, 7, 44)
    M = P.plan(n)['M']
    r = _rank_desc(x)
    x = x - x[r[M]] + 0.3
    c = x[r[M]]
    up = np.nextafter(c, np.inf)
    x[r[M - 40:M]] = up
    mx = x.max()
    assert up - mx == c - mx and up > c
    return x


def _minus_inf(n):
    x = _t_ratio(n, 5, 7, 45)
    x[[3, n // 2, n - 1]] = -np.inf
    return x


def _with(x, pos, val):
    x = x.copy()
    x[pos] = val
    return x


CONTENT_N = 4000


def _content_cases():
    n = CONTENT_N
    base = _t_ratio(n, 5, 7, 46)
    return {
        'k_below_third': _t_ratio(n, 50, 5, 1),
        'k_third_to_0.7': _t_ratio(n, 3, 30, 3),
        'k_above_1_clipped': _capped_pareto(n, 2),
        'all_equal': np.full(n, -3.25),
        'tie_straddle': _tie_straddle(n),
        'signed_zeros': _signed_zeros(n),
        'huge_pm_1e308': _huge_pm(n),
        'huge_1e308': _with(base, 17, 1e308),
        'pos_inf': _with(base, [0, 777], np.inf),
        'nan_first': _with(base, 0, np.nan),
        'nan_last': _with(base, n - 1, -np.nan),
        'minus_inf': _minus_inf(n),
        'below_floor': _floor(n),
        'ulp_above_cutoff': _ulp_above(n),
        'neighbour': base,
    }


def test_column_contents(psis, vo):
    cases = _content_cases()
    names = list(cases)
    refs = _check_all(psis, [cases[k] for k in names], 1.0, 'contents')
    ref = dict(zip(names, refs))
    # the cases reach what they are named for
    assert ref['k_below_third']['k'] < 1.0 / 3.0
    assert 1.0 / 3.0 <= ref['k_third_to_0.7']['k'] < 0.7
    assert ref['k_above_1_clipped']['k'] > 1.0
    assert np.sum(ref['k_above_1_clipped']['out'] == -ref['k_above_1_clipped']['lse']) > 1    # several clipped to 0
    assert ref['all_equal']['n2'] == 0 and ref['below_floor']['xcut'] == LOG_TINY and ref['below_floor']['n2'] == 100
    assert np.isnan(ref['nan_first']['lse']) and np.isposinf(ref['nan_first']['k'])
    assert ref['neighbour']['n2'] > 4 and np.isfinite(ref['neighbour']['k'])


def test_small_tails(psis):
    """n2 <= 4 (k-hat +inf, nothing smoothed) and the smallest columns."""
    for n in (2, 3, 5, 9, 20):
        cols = [P.small_case(kind, n) for kind in P.SMALL_KINDS] + [psis_case('tiny_20')[:n]]
        refs = _check_all(psis, cols, 1.0, ('small', n))
        assert all(r['n2'] <= 4 for r in refs)


# ---- shapes --------------------------------------------------------------------------------------------------------
REFFS = (1.0, 0.3, 0.05)


@pytest.mark.parametrize('reff', REFFS)
def test_shapes(psis, vb, reff):
    max_n = psis.psis_batch_max_n(reff)
    assert max_n > 1000 and max_n == vb._lib.lib.vb_psis_batch_max_n(reff)
    if reff == 1.0:
        assert 20000 < max_n < 30000
    for n in (2, 3, 5, 31, 32, 33, 1000, 4000, max_n - 1, max_n):
        cols = [_t_ratio(n, 5, 7, 50 + n % 97), _t_ratio(n, 3, 30, 51), _tie_straddle(n, reff) if n > 40 else
                P.small_case('three_values', n)]
        refs = _check_all(psis, cols, reff, ('shape', n, reff))
        if n in (1000, 4000) and reff == 0.05:
            assert refs[0]['M'] == math.ceil(0.2 * n)          # the 0.2 n bound binds


def test_fallback_above_max_n(psis, vb):
    """One past the shared-memory limit: the C ABI refuses, and 2-D psislw takes the one-column pipeline."""
    n = psis.psis_batch_max_n(1.0) + 1
    cols = [_t_ratio(n, 5, 7, 60), _t_ratio(n, 3, 30, 61)]
    with pytest.raises(NotImplementedError):
        _run(psis, cols)
    X = np.stack(cols, axis=1)
    out, k = vb.psislw(X)
    assert out.flags.f_contiguous
    for j, x in enumerate(cols):
        ref = P.oracle(x)
        _close(k[j], ref['k'], 'k')
        np.testing.assert_allclose(out[:, j], ref['out'], rtol=TOL, atol=TOL)


# ---- grid and memory edges ---------------------------------------------------------------------------------------
def _mixed(n, m, seed):
    rs = np.random.RandomState(seed)
    X = rs.standard_t(3, size=(n, m)) * rs.uniform(0.2, 3.0, size=m)
    return X


@pytest.mark.parametrize('m', [1, 7, 70000])
def test_grid_edges(psis, m):
    n = 64
    X = _mixed(n, m, 70 + m)
    out, k, r, loo = _run(psis, list(X.T))
    check = range(m) if m <= 7 else list(range(0, m, 997)) + list(range(m - 50, m))
    for j in check:
        _check_col(X[:, j], 1.0, r[j], k[j], out[:, j], loo[j], ('grid', m, j))


def test_offset_and_leading_dimension(psis):
    """ld > n with lw starting one double into its buffer; out with its own leading dimension and sentinels."""
    n, m, ld, ldo = 1000, 9, 1003, 1005
    X = _mixed(n, m, 80)
    buf = torch.full((ld * m + 1,), 7.5, dtype=torch.float64, device='cuda')
    lw = torch.as_strided(buf, (n, m), (1, ld), 1)
    lw.copy_(torch.from_numpy(X))
    before = buf.clone()
    obuf = torch.full((ldo * m + 16,), float('nan'), dtype=torch.float64, device='cuda')
    obuf[ldo * m:] = torch.arange(16, dtype=torch.float64) + 1234.5
    out = torch.as_strided(obuf, (n, m), (1, ldo), 0)
    _, k, r, loo = psis.psislw_batch_device(lw, out, 1.0, want_loo=True, want_result=True)
    ob = obuf.cpu().numpy()
    assert torch.equal(buf, before)                                        # the input is read only
    assert np.array_equal(ob[ldo * m:], np.arange(16) + 1234.5)            # nothing after the last column
    gaps = ob[:ldo * m].reshape(m, ldo)[:, n:]
    assert np.isnan(gaps).all()                                            # nor between columns
    o = out.cpu().numpy()
    for j in range(m):
        _check_col(X[:, j], 1.0, r[j].cpu().numpy(), float(k[j]), o[:, j], float(loo[j]), ('ld', j))


def test_past_2_31_entries(psis):
    """m * ld > 2^31: the last columns are read and written at 64-bit offsets."""
    n, ld = 1000, 1024
    m = (2 ** 31) // ld + 4
    X = torch.empty((m, ld), dtype=torch.float64, device='cuda')
    X.normal_(generator=torch.Generator(device='cuda').manual_seed(90))
    cols = {j: _t_ratio(n, 3, 30, 91 + j % 5) for j in (0, 1, m - 3, m - 2, m - 1)}
    for j, x in cols.items():
        X[j, :n] = torch.from_numpy(x)
    lw = X.t()[:n]                                                         # n x m, leading dimension 1024
    _, k, r, loo = psis.psislw_batch_device(lw, lw, 1.0, want_loo=True, want_result=True)
    for j, x in cols.items():
        _check_col(x, 1.0, r[j].cpu().numpy(), float(k[j]), X[j, :n].cpu().numpy(), None, ('2^31', j))
    del X, lw
    torch.cuda.empty_cache()


# ---- output modes and determinism --------------------------------------------------------------------------------
def test_output_modes_bitwise(psis):
    cases = _content_cases()
    cols = list(cases.values()) + [_t_ratio(CONTENT_N, 4, 9, 100 + j) for j in range(20)]
    X = np.stack(cols, axis=1)
    t = torch.from_numpy(np.ascontiguousarray(X.T)).cuda().t()
    runs = []
    for _ in range(3):
        o = torch.empty_like(t)
        runs.append(psis.psislw_batch_device(t, o, 1.0, want_loo=True, want_result=True))
    b = [tuple(x.cpu().numpy().tobytes() for x in run) for run in runs]
    assert b[0] == b[1] == b[2]                                            # three bitwise-equal repeats
    _, k0, r0, l0 = psis.psislw_batch_device(t, None, 1.0, want_loo=True, want_result=True)
    assert k0.cpu().numpy().tobytes() == b[0][1] and l0.cpu().numpy().tobytes() == b[0][3]
    assert r0.cpu().numpy().tobytes() == b[0][2]
    # out aliasing lw: the same bits as a separate output
    t2 = t.clone()
    _, k2, _, l2 = psis.psislw_batch_device(t2, t2, 1.0, want_loo=True)
    assert t2.cpu().numpy().tobytes() == runs[0][0].cpu().numpy().tobytes()
    assert k2.cpu().numpy().tobytes() == b[0][1] and l2.cpu().numpy().tobytes() == b[0][3]
    assert t.t().contiguous().cpu().numpy().tobytes() == np.ascontiguousarray(X.T).tobytes()   # lw untouched, bitwise


# ---- psisloo and 2-D psislw ---------------------------------------------------------------------------------------
_loo_ref = {}


def _loo_problem(vo):
    if 'll' not in _loo_ref:
        rs = np.random.RandomState(110)
        n, m = 4000, 10000
        ll = -np.abs(rs.standard_t(4, size=(n, m))) * rs.uniform(0.1, 2.0, size=m)
        ll[:, 7] = -_capped_pareto(n, 3)                                     # a smoothed, clipped column
        with np.errstate(all='ignore'):
            _loo_ref['ll'] = ll
            _loo_ref['ref'] = vo.psisloo(ll)
    return _loo_ref['ll'], _loo_ref['ref']


def test_psisloo_numpy(vb, vo):
    ll, (loo0, loos0, ks0) = _loo_problem(vo)
    keep = ll.copy()
    loo, loos, ks = vb.psisloo(ll)
    assert np.array_equal(ll, keep)
    assert isinstance(loo, float) and isinstance(loos, np.ndarray) and isinstance(ks, np.ndarray)
    _close(loo, loo0, 'loo')
    np.testing.assert_allclose(loos, loos0, rtol=TOL, atol=0)
    assert np.array_equal(np.isinf(ks), np.isinf(ks0))
    fin = np.isfinite(ks0)
    np.testing.assert_allclose(ks[fin], ks0[fin], rtol=TOL, atol=1e-300)
    loo_f, _, _ = vb.psisloo(np.asfortranarray(ll))
    assert loo_f == loo


def test_psisloo_cuda(vb, vo):
    ll, (loo0, loos0, ks0) = _loo_problem(vo)
    t = torch.from_numpy(ll).cuda()
    keep = t.clone()
    loo, loos, ks = vb.psisloo(t)
    assert torch.equal(t, keep)
    assert loo.is_cuda and loo.dim() == 0 and loos.is_cuda and ks.is_cuda
    _close(float(loo), loo0, 'loo')
    np.testing.assert_allclose(loos.cpu().numpy(), loos0, rtol=TOL, atol=0)
    k = ks.cpu().numpy()
    fin = np.isfinite(ks0)
    assert np.array_equal(np.isinf(k), np.isinf(ks0))
    np.testing.assert_allclose(k[fin], ks0[fin], rtol=TOL, atol=1e-300)
    # an F-ordered tensor and a column slice (leading dimension > n) give the same bits
    loo_f, loos_f, _ = vb.psisloo(t.t().contiguous().t())
    assert torch.equal(loos_f, loos)
    _, loos_s, _ = vb.psisloo(t[:, 3:9])
    assert torch.equal(loos_s, loos[3:9])


def test_psislw_2d_forms(vb, vo):
    n, m = 1000, 20
    X = _mixed(n, m, 120)
    X[:, 3] = _capped_pareto(n, 4)
    refs = [vo.psislw_1d(X[:, j]) for j in range(m)]
    o_ref = np.stack([r[0] for r in refs], axis=1)
    k_ref = np.array([r[1] for r in refs])

    def check(out, k):
        np.testing.assert_allclose(out, o_ref, rtol=TOL, atol=TOL)
        np.testing.assert_allclose(k, k_ref, rtol=TOL, atol=1e-300)

    for order in ('C', 'F'):
        a = np.array(X, order=order)
        out, k = vb.psislw(a)
        assert isinstance(out, np.ndarray) and out.flags.f_contiguous and isinstance(k, np.ndarray)
        check(out, k)
        assert np.array_equal(a, X)
        out, k = vb.psislw(a, overwrite_lw=True)
        check(out, k)
        if order == 'F':
            assert out is a                          # F-contiguous float64: smoothed in place
        else:
            assert np.array_equal(a, X)
    for layout in ('C', 'F'):
        t = torch.from_numpy(X).cuda() if layout == 'C' else torch.from_numpy(np.ascontiguousarray(X.T)).cuda().t()
        out, k = vb.psislw(t)
        assert out.is_cuda and out.data_ptr() != t.data_ptr()
        check(out.cpu().numpy(), k)
        assert np.array_equal(t.cpu().numpy(), X)
        out, k = vb.psislw(t, overwrite_lw=True)
        assert out is t
        check(t.cpu().numpy(), k)


# ---- C ABI errors -------------------------------------------------------------------------------------------------
def test_cabi_errors(vb, psis):
    L = vb._lib
    lib = L.lib
    n, m = 100, 4
    lw = torch.randn(m, n, dtype=torch.float64, device='cuda')
    out = torch.full((m, n), 5.5, dtype=torch.float64, device='cuda')
    khat = torch.full((m,), 5.5, dtype=torch.float64, device='cuda')
    res = torch.full((m, 16), 5.5, dtype=torch.float64, device='cuda')
    loo = torch.full((m,), 5.5, dtype=torch.float64, device='cuda')
    P_ = lambda t: ctypes.c_void_p(t.data_ptr())                                     # noqa: E731
    base = dict(lw=P_(lw), ld=n, n=n, m=m, reff=1.0, out=P_(out), ldo=n, khat=P_(khat), res=P_(res), loo=P_(loo))

    def call(**kw):
        a = dict(base, **kw)
        return lib.vb_psislw_batch_f64(a['lw'], a['ld'], a['n'], a['m'], a['reff'], a['out'], a['ldo'], a['khat'],
                                       a['res'], a['loo'], L.stream())
    max_n = lib.vb_psis_batch_max_n(1.0)
    bad = [(dict(n=1, ld=1, ldo=1), L.VB_ERR_INVALID_ARG), (dict(n=0), L.VB_ERR_INVALID_ARG),
           (dict(m=-1), L.VB_ERR_INVALID_ARG), (dict(ld=n - 1), L.VB_ERR_INVALID_ARG),
           (dict(ldo=n - 1), L.VB_ERR_INVALID_ARG), (dict(reff=0.0), L.VB_ERR_INVALID_ARG),
           (dict(reff=-1.0), L.VB_ERR_INVALID_ARG), (dict(reff=float('nan')), L.VB_ERR_INVALID_ARG),
           (dict(lw=None), L.VB_ERR_INVALID_ARG), (dict(khat=None), L.VB_ERR_INVALID_ARG),
           (dict(n=max_n + 1, ld=max_n + 1, ldo=max_n + 1, m=1), L.VB_ERR_UNSUPPORTED)]
    for kw, code in bad:
        assert call(**kw) == code, kw
        torch.cuda.synchronize()
        for t in (out, khat, res, loo):
            assert bool((t == 5.5).all()), kw                                         # nothing written
    assert lib.vb_psis_batch_max_n(0.0) == 0 and lib.vb_psis_batch_max_n(-1.0) == 0
    assert lib.vb_psis_batch_max_n(0.05) < lib.vb_psis_batch_max_n(0.3) <= max_n
    assert call(m=0) == L.VB_OK                                                      # m = 0: a no-op
    torch.cuda.synchronize()
    assert bool((khat == 5.5).all())
    assert call() == L.VB_OK
    _, k, _, _ = psis.psislw_batch_device(lw.t(), None, 1.0)
    assert torch.equal(khat, k)
