"""The exact GLM kernels element by element, through the C ABI: vb_glm_sweep_f64 against a float64 reference under
per-element worst-case bounds (tests/_glm_f64_ref.py) at d, S and N around its plan regimes, tiles, super-chunks and
CTA wave, in every mode; vb_glm_link_f64 and vb_glm_point_f64 against mpmath per element; the Hessian SYRK against
long double.  Bitwise reproducibility is required wherever the kernels promise fixed-order sums."""
import numpy as np
import pytest
import torch

from _glm_f64_ref import (CASES, LINK_ID, Reference, alpha_weights, case_links, case_seed, ll_rtol, make_case, mp_link,
                          plan, ratios)

pytestmark = pytest.mark.gpu
SENT = -7.25e77
PAD = 8


def _L():
    from viabel_b200 import _lib
    return _lib


def _dev(a):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device='cuda')


def _eq(a, b):
    return a is not None and b is not None and np.array_equal(a, b)


def _padded(a, offset=0):
    """a on the device followed by PAD sentinels, starting `offset` doubles into its buffer."""
    a = np.asarray(a, dtype=np.float64).ravel()
    buf = torch.full((offset + a.size + PAD,), SENT, dtype=torch.float64, device='cuda')
    buf[offset:offset + a.size] = _dev(a)
    return buf, buf[offset:]


def sweep(X, y, theta, base, link, w=None, aux=None, want_grad=1, ldx=None, xoff=0, ws_fill=0xFF, ws_bytes=None):
    """One vb_glm_sweep_f64 call; X stored with leading dimension ldx (NaN padding) `xoff` doubles into its buffer.
    Returns (rc, ll, gmu, ge); sentinels after each output must survive, gradient outputs stay untouched without
    want_grad."""
    L = _L()
    N, d = X.shape
    S = theta.shape[0]
    ldx = d if ldx is None else ldx
    Xp = np.full((N, ldx), np.nan)
    Xp[:, :d] = X
    xbuf = torch.full((xoff + max(Xp.size, 1),), np.nan, dtype=torch.float64, device='cuda')
    xbuf[xoff:xoff + Xp.size] = _dev(Xp.ravel())
    Xd = xbuf[xoff:]
    nb = L.lib.vb_glm_sweep_workspace_bytes(N, d, S) if ws_bytes is None else ws_bytes
    ws = torch.empty(max(nb, 1), dtype=torch.uint8, device='cuda')
    ws.fill_(ws_fill)
    outs = [torch.full((n + PAD,), SENT, dtype=torch.float64, device='cuda') for n in (S, d, d)]
    yd, th = _dev(y if N else np.zeros(1)), _dev(theta)
    bs = _dev(base) if (want_grad and base is not None) else None
    wd = None if w is None else _dev(w)
    ad = None if aux is None else _dev(aux)
    rc = L.lib.vb_glm_sweep_f64(L.ptr(Xd), ldx, L.ptr(yd), N, d, LINK_ID[link], L.ptr(th), L.ptr(bs), L.ptr(wd),
                                L.ptr(ad), S, want_grad, L.ptr(outs[0]), L.ptr(outs[1]) if want_grad else None,
                                L.ptr(outs[2]) if want_grad else None, L.ptr(ws), nb, L.stream())
    torch.cuda.synchronize()
    o = [t.cpu().numpy() for t in outs]
    if rc != 0:
        assert all(np.all(a == SENT) for a in o), 'outputs written by a failing call'
        return rc, None, None, None
    assert np.all(o[0][S:] == SENT), 'll written past S'
    if want_grad:
        for a in o[1:]:
            assert np.all(a[d:] == SENT), 'gradient written past d'
        return rc, o[0][:S], o[1][:d], o[2][:d]
    assert np.all(o[1] == SENT) and np.all(o[2] == SENT), 'gradient written without want_grad'
    return rc, o[0][:S], None, None


def run_case(N, d, S):
    """Every mode of one shape; returns {link/mode: {output: err / bound}}."""
    res = {}
    for li, link in enumerate(case_links(N, S)):
        X, y, theta, base, aux = make_case(N, d, S, link, case_seed(N, d, S))
        ax = aux if link == 'gaussian' else None
        ref = Reference(X, y, theta, base, link, aux=aux)
        rc, ll, gmu, ge = sweep(X, y, theta, base, link, aux=ax, ws_fill=0)
        assert rc == 0, _L().last_error()
        res[link] = ratios(ref, ll, gmu, ge)
        r0 = sweep(X, y, theta, None, link, aux=ax, want_grad=0)
        assert r0[0] == 0 and _eq(r0[1], ll), 'want_grad = 0 changes ll'
        r1 = sweep(X, y, theta, base, link, w=np.ones(S), aux=ax)
        assert _eq(r1[1], ll) and _eq(r1[2], gmu) and _eq(r1[3], ge), 'all-ones weights differ from w = NULL'
        w = alpha_weights(S, S + d)
        refw = Reference(X, y, theta, base, link, w=w, aux=aux)
        rw = sweep(X, y, theta, base, link, w=w, aux=ax)
        assert _eq(rw[1], ll), 'weights change ll'
        res[link + '/weighted'] = ratios(refw, rw[1], rw[2], rw[3])
        if li == 0:
            # NaN-filled workspace (the default fill), repeated; wide and unaligned X: the scalar staging path
            for kw in ({}, {}, {'ldx': d + 1}, {'ldx': d + 8}, {'xoff': 1}, {'ldx': d + 8, 'xoff': 1}):
                r2 = sweep(X, y, theta, base, link, aux=ax, **kw)
                assert _eq(r2[1], ll) and _eq(r2[2], gmu) and _eq(r2[3], ge), ('not bitwise equal', kw)
    return res


def _check(res, tag):
    print('%s: %s' % (tag, ', '.join('%s/%s %.3g' % (m, o, v) for m, r in res.items() for o, v in r.items())))
    for mode, r in res.items():
        for out, v in r.items():
            assert v <= 1.0, (tag, mode, out, v)


@pytest.mark.parametrize('N,d,S', CASES)
def test_sweep_elementwise(N, d, S):
    _check(run_case(N, d, S), (N, d, S))


def test_sweep_edges():
    """d = 2897 is rejected without writing anything; N = 0 gives zeros; a workspace one byte short is rejected; the
    workspace size follows the plan (per-warp ge rows in global memory exactly where they do not fit on chip)."""
    L = _L()
    X, y, theta, base, _ = make_case(3, 2897, 4, 'logistic', 1)
    assert L.lib.vb_glm_sweep_workspace_bytes(3, 2897, 4) == 0
    rc = sweep(X, y, theta, base, 'logistic', ws_bytes=1 << 20)[0]
    assert rc == L.VB_ERR_UNSUPPORTED
    for d in (9, 2896):
        X, y, theta, base, _ = make_case(0, d, 17, 'logistic', 2)
        rc, ll, gmu, ge = sweep(X, y, theta, base, 'logistic')
        assert rc == 0 and np.all(ll == 0) and np.all(gmu == 0) and np.all(ge == 0)
    X, y, theta, base, _ = make_case(100, 40, 17, 'logistic', 3)
    assert sweep(X, y, theta, base, 'logistic', ws_bytes=L.lib.vb_glm_sweep_workspace_bytes(100, 40, 17) - 1)[0] \
        == L.VB_ERR_WORKSPACE
    sms = L.lib.vb_device_sm_count()
    ws = lambda d: L.lib.vb_glm_sweep_workspace_bytes(100000, d, 16)
    rows = lambda d: sms * 16 * (-(-d // 8) * 8) * 8
    assert ws(577) - ws(576) >= rows(577) and ws(865) - ws(864) >= rows(865)
    assert ws(864) < ws(832)


@pytest.mark.parametrize('d', [512, 1024])
def test_fused_step_f64_bitwise(d):
    """The f64 fused step (the exact leg of the benchmark) twice from the same state, and eager against graph replay:
    bitwise equal (d = 1024 accumulates ge in per-warp global rows)."""
    import viabel_b200 as vb
    from viabel_b200.engine import FusedStep
    N, S = 20011, 256
    X, y, theta, base, _ = make_case(N, d, S, 'logistic', 7, saturate=False)
    model = vb.LogisticRegression(X, y, prior_scale=10.0)
    assert model.path == 'f64'
    rs = np.random.RandomState(d)
    p0 = np.concatenate([rs.randn(d) / np.sqrt(d), -1.0 + 0.1 * rs.randn(d)])
    outs = []
    for use_graph in (False, False, True, True):
        eng = FusedStep(vb.ExclusiveKL(vb.MFGaussian(d), model, S), None, inject_base=True)
        eng.set_param(p0)
        eng.base.copy_(_dev(base))
        eng.run(1, use_graph=use_graph)
        torch.cuda.synchronize()
        outs.append(eng.out.cpu().numpy().copy())
        del eng
    for o in outs[1:]:
        assert np.array_equal(o, outs[0])


# ---- vb_glm_link_f64 ------------------------------------------------------------------------------------------------
def _grid():
    g = np.logspace(-3, 4, 400)
    special = [0.0, -0.0, 5e-324, -5e-324, 1e-310, -1e-310, 2.2e-308, -2.2e-308, -37.5, -37.0, -20.0, -6.0, -5.99,
               -6.01, 8.0, 20.0, 36.0, 40.0, 745.0, -745.0, 1e4, -1e4]
    return np.concatenate([-g, g, special])


def link_call(A, y, link, prev):
    L = _L()
    Nc, S = A.shape
    Ad, yd, lld = _dev(A), _dev(y), _dev(prev)
    ws = torch.empty(L.lib.vb_glm_link_workspace_bytes(Nc, S), dtype=torch.uint8, device='cuda').fill_(0xFF)
    rc = L.lib.vb_glm_link_f64(L.ptr(Ad), L.ptr(yd), Nc, S, LINK_ID[link], L.ptr(lld), L.ptr(ws), ws.numel(),
                               L.stream())
    torch.cuda.synchronize()
    assert rc == 0, L.last_error()
    return Ad.cpu().numpy(), lld.cpu().numpy()


def _close(got, want, rtol, atol=2e-323):
    return np.abs(got - want) <= rtol * np.abs(want) + atol


@pytest.mark.parametrize('link', ['logistic', 'probit'])
def test_link_step_grid_vs_mpmath(link):
    """One row of a over [-1e4, 1e4] with +-0 and subnormals, y = +1 and -1: ll (a single-element column sum is the
    element itself; a few ulps times its condition number) and y dl to a few ulps of the mpmath values."""
    a = _grid()
    m = np.array([mp_link(v, link) for v in a])
    for yv in (1.0, -1.0):
        out, ll = link_call(a[None, :], np.array([yv]), link, np.zeros(a.size))
        bad = ~_close(ll, m[:, 0], ll_rtol(a, m[:, 0], m[:, 1]))
        assert not bad.any(), ('ll', a[bad][:8], ll[bad][:8], m[bad, 0][:8])
        bad = ~_close(out[0], yv * m[:, 1], 1e-14)
        assert not bad.any(), ('y dl', yv, a[bad][:8], out[0][bad][:8], m[bad, 1][:8])


@pytest.mark.parametrize('Nc', [511, 512, 513])
@pytest.mark.parametrize('S', [31, 32, 33])
def test_link_step_shapes(Nc, S):
    """Row blocks of 512 and column blocks of 32 at their edges; ll_accum accumulates onto its contents."""
    from _glm_f64_ref import link_terms
    rs = np.random.RandomState(Nc + S)
    for link in ('logistic', 'probit'):
        A = 8.0 * rs.randn(Nc, S)
        y = np.where(rs.rand(Nc) < 0.5, 1.0, -1.0)
        prev = 1000.0 * rs.randn(S)
        out, ll = link_call(A, y, link, prev)
        l0, r0, _, _ = link_terms(A, np.ones(Nc), link)
        assert np.all(_close(out, y[:, None] * r0, 1e-14))
        want = prev + l0.sum(axis=0)
        assert np.all(np.abs(ll - want) <= 1e-15 * (Nc + 2) * (np.abs(prev) + np.abs(l0).sum(axis=0)))


def test_link_step_past_65535_row_blocks():
    """S = 33 (two column blocks) and Nc = 2^24 + 513 rows: 65 540 CTAs.  A repeats one 512-row pattern, so each column
    sum is known from the pattern; rows in the first, the last and past the 65 535th block are checked."""
    from _glm_f64_ref import link_terms
    S, Nc = 33, (1 << 24) + 513
    rs = np.random.RandomState(9)
    pat = 6.0 * rs.randn(512, S)
    ypat = np.where(rs.rand(512) < 0.5, 1.0, -1.0)
    reps = -(-Nc // 512)
    L = _L()
    A = _dev(pat).repeat(reps, 1)[:Nc].contiguous()
    y = _dev(ypat).repeat(reps)[:Nc].contiguous()
    ll = torch.zeros(S, dtype=torch.float64, device='cuda')
    ws = torch.empty(L.lib.vb_glm_link_workspace_bytes(Nc, S), dtype=torch.uint8, device='cuda')
    assert L.lib.vb_glm_link_f64(L.ptr(A), L.ptr(y), Nc, S, 0, L.ptr(ll), L.ptr(ws), ws.numel(), L.stream()) == 0
    torch.cuda.synchronize()
    l0, r0, _, _ = link_terms(pat, np.ones(512), 'logistic')
    full, rest = divmod(Nc, 512)
    want = full * l0.sum(axis=0) + l0[:rest].sum(axis=0)
    got = ll.cpu().numpy()
    # each column: 64-row thread sums, 8 row groups, then 32 770 block partials added in order
    bound = 2.0 ** -52 * (Nc / 512.0 + 80.0) * (full + 1) * np.abs(l0).sum(axis=0)
    assert np.all(np.abs(got - want) <= bound), np.max(np.abs(got - want) / bound)
    for lo in (0, 32767 * 512 - 512, Nc - 1024):       # row block 32 767 holds CTAs 65 534 and 65 535
        blk = A[lo:lo + 1024].cpu().numpy()
        idx = (np.arange(lo, lo + 1024) % 512)
        assert np.all(_close(blk, ypat[idx, None] * r0[idx], 1e-14)), lo
    del A


# ---- vb_glm_point_f64 -----------------------------------------------------------------------------------------------
def point_call(X, y, theta, link, V=None, hessian=False, want_ll=True, N=None, ldx=None):
    L = _L()
    Xd = X if torch.is_tensor(X) else _dev(X)
    N = Xd.shape[0] if N is None else N
    d = theta.size
    K = 0 if V is None else V.shape[0]
    nb = L.lib.vb_glm_point_workspace_bytes(N, d, K, int(hessian))
    ws = torch.empty(max(nb, 8), dtype=torch.uint8, device='cuda').fill_(0xFF)
    g_buf, g = _padded(np.zeros(d))
    hv_buf, hv = _padded(np.zeros(max(K, 1) * d))
    H_buf, H = _padded(np.zeros(d * d if hessian else 1))
    ll_buf, ll = _padded(np.zeros(1))
    Vd = None if V is None else _dev(V)
    yd, thd = _dev(y), _dev(theta)          # held until the call has run: the allocator reuses freed blocks
    rc = L.lib.vb_glm_point_f64(L.ptr(Xd), d if ldx is None else ldx, L.ptr(yd), N, d, LINK_ID[link],
                                L.ptr(thd), L.ptr(Vd), K, L.ptr(ll) if want_ll else None, L.ptr(g),
                                L.ptr(hv) if K else None, L.ptr(H) if hessian else None, L.ptr(ws), nb, L.stream())
    torch.cuda.synchronize()
    if rc != 0:
        return rc, None
    res = {}
    for name, buf, n in (('g', g_buf, d), ('hv', hv_buf, K * d), ('H', H_buf, d * d if hessian else 0),
                         ('ll', ll_buf, 1)):
        a = buf.cpu().numpy()
        assert np.all(a[-PAD:] == SENT), name + ' written past its end'
        res[name] = a[:n]
    res['hv'] = res['hv'].reshape(K, d)
    res['H'] = res['H'].reshape(d, d) if hessian else None
    return rc, res


@pytest.mark.parametrize('link', ['logistic', 'probit'])
def test_point_per_row_vs_mpmath(link):
    """X = I (N = d = 2048), theta_n = a_n y_n: grad_n = y_n dl(a_n), hvp_n = -c(a_n) v_n with v = 1, H_nn = -c(a_n),
    each a single product, against mpmath over a in [-1e4, 1e4].  dl to 1e-14, c to 1e-12 relative (where they are
    normal numbers)."""
    d = 2048
    g = np.logspace(-2, 4, 1000)
    a = np.concatenate([-g, g, [0.0, -6.0, -6.01, -5.99, -20.0, -37.0, -37.5, -700.0, -740.0, 8.0, 20.0, 40.0]])
    a = np.concatenate([a, np.linspace(-50, 50, d - a.size)])
    rs = np.random.RandomState(4)
    y = np.where(rs.rand(d) < 0.5, 1.0, -1.0)
    theta = a * y
    X = torch.eye(d, dtype=torch.float64, device='cuda')
    rc, res = point_call(X, y, theta, link, V=np.ones((1, d)), hessian=True)
    assert rc == 0, _L().last_error()
    m = np.array([mp_link(v, link) for v in a])
    bad = ~_close(res['g'], y * m[:, 1], 1e-14)
    assert not bad.any(), ('grad', a[bad][:8], res['g'][bad][:8], (y * m[:, 1])[bad][:8])
    for name, got in (('hvp', res['hv'][0]), ('H diag', np.diag(res['H']))):
        # r is subnormal beyond a ~ 37.5 (probit): there only 2^-1032 absolute
        bad = ~_close(-got, m[:, 2], 1e-12, 2.0 ** -1032)
        assert not bad.any(), (name, a[bad][:8], -got[bad][:8], m[bad, 2][:8])
    assert np.all(res['H'] - np.diag(np.diag(res['H'])) == 0)
    want_ll = sum(r[0] for r in m)
    assert abs(res['ll'][0] - want_ll) <= 1e-13 * np.sum(np.abs(m[:, 0])) + 1e-300


def _point_ref(X, y, theta, link, V):
    """grad, HVPs and Hessian in long double from float64 links, and worst-case bounds."""
    from _glm_f64_ref import link_terms, U
    Xl = X.astype(np.longdouble)
    a = (Xl @ theta.astype(np.longdouble)).astype(np.float64)
    ll, r, c, _ = link_terms(a[:, None], y, link)
    ll, r, c = ll[:, 0], r[:, 0], c[:, 0]
    aX = np.abs(X)
    da = 16 * U * (aX @ np.abs(theta))
    N = X.shape[0]
    ns = N / 256.0 + 600.0
    g = (Xl.T @ r.astype(np.longdouble)).astype(np.float64)
    gb = aX.T @ (c * da + 8 * U * np.abs(r)) + U * ns * (aX.T @ np.abs(r))
    out = {'g': (g, gb), 'll': (np.sum(ll.astype(np.longdouble)), np.sum(np.abs(ll)) * U * (8 + ns))}
    if V is not None and V.shape[0]:
        t = (Xl @ V.T.astype(np.longdouble)).astype(np.float64)      # [N, K]
        tb = 16 * U * (aX @ np.abs(V).T)
        hv = -(Xl.T @ (c[:, None] * t).astype(np.longdouble)).astype(np.float64).T
        hb = (aX.T @ ((da[:, None] * (c + 1.0)[:, None]) * np.abs(t) + c[:, None] * tb
                      + 8 * U * c[:, None] * np.abs(t)) + U * ns * (aX.T @ (c[:, None] * np.abs(t)))).T
        out['hv'] = (hv, hb)
    out['c'], out['da'] = c, da
    return out


def _within(got, want, bound):
    return np.all(np.abs(got - want) <= bound + 1e-300)


POINT_CASES = [(31, 1, 0), (32, 255, 1), (33, 256, 2), (63, 257, 3), (9473, 2047, 4), (1000, 2048, 8),
               (9504, 256, 8), (2 * 148 * 32 + 1, 1, 4), (65, 257, 0), (4097, 100, 3)]


@pytest.mark.parametrize('N,d,K', POINT_CASES)
def test_point_general(N, d, K):
    """grad and K HVPs at d around 8 columns per thread and N at 32-row tile edges and past 2 x 148 tiles, both links,
    against long double under a worst-case bound; out_ll NULL gives the same gradient bitwise."""
    rs = np.random.RandomState(N + d + K)
    X = rs.randn(N, d)
    y = np.where(rs.rand(N) < 0.5, 1.0, -1.0)
    theta = rs.randn(d) * 1.5 / np.sqrt(d)
    X[N // 2] *= 300.0                                         # a saturated row
    V = rs.randn(K, d) if K else None
    for link in ('logistic', 'probit'):
        rc, res = point_call(X, y, theta, link, V=V)
        assert rc == 0, _L().last_error()
        ref = _point_ref(X, y, theta, link, V)
        assert _within(res['g'], *ref['g']), (link, np.max(np.abs(res['g'] - ref['g'][0]) / ref['g'][1]))
        assert abs(res['ll'][0] - float(ref['ll'][0])) <= ref['ll'][1] + 1e-300
        if K:
            assert _within(res['hv'], *ref['hv']), (link, np.max(np.abs(res['hv'] - ref['hv'][0]) / ref['hv'][1]))
        rc, res2 = point_call(X, y, theta, link, V=V, want_ll=False)
        assert rc == 0 and _eq(res2['g'], res['g']) and _eq(res2['hv'], res['hv'])


@pytest.mark.parametrize('N,d', [(1000, 100), (3001, 257), (33, 65)])
def test_point_hessian_vs_long_double(N, d):
    """The weighted SYRK Hessian at N not a multiple of 32 and d not a multiple of 64: element by element against long
    double, bitwise symmetric; the same Hessian on repeat."""
    from _glm_f64_ref import U
    rs = np.random.RandomState(N * d)
    X = rs.randn(N, d)
    y = np.where(rs.rand(N) < 0.5, 1.0, -1.0)
    theta = rs.randn(d) * 2.0 / np.sqrt(d)
    for link in ('logistic', 'probit'):
        rc, res = point_call(X, y, theta, link, hessian=True)
        assert rc == 0, _L().last_error()
        ref = _point_ref(X, y, theta, link, None)
        c, da = ref['c'], ref['da']
        Xl = X.astype(np.longdouble)
        H = -(Xl.T @ (c.astype(np.longdouble)[:, None] * Xl)).astype(np.float64)
        aX = np.abs(X)
        B = aX.T @ ((da + 8 * U * c)[:, None] * aX) + U * (N + 64) * (aX.T @ (c[:, None] * aX))
        assert _within(res['H'], H, B), (link, np.max(np.abs(res['H'] - H) / B))
        assert np.array_equal(res['H'], res['H'].T)
        rc, again = point_call(X, y, theta, link, hessian=True)
        assert _eq(again['H'], res['H'])


def test_point_edges():
    """K = 5..7 and d = 2049 are rejected; N = 0 gives zeros (Hessian included)."""
    L = _L()
    rs = np.random.RandomState(1)
    X, y = rs.randn(40, 16), np.ones(40)
    for K in (5, 6, 7):
        assert point_call(X, y, rs.randn(16), 'logistic', V=rs.randn(K, 16))[0] == L.VB_ERR_UNSUPPORTED
    assert point_call(rs.randn(4, 2049), np.ones(4), rs.randn(2049), 'probit')[0] == L.VB_ERR_UNSUPPORTED
    rc, res = point_call(X, y, rs.randn(16), 'probit', V=rs.randn(2, 16), hessian=True, N=0)
    assert rc == 0
    assert np.all(res['g'] == 0) and np.all(res['hv'] == 0) and np.all(res['H'] == 0) and res['ll'][0] == 0
