"""GPU: MultivariateT's default sqrtm mode, theta = mu + (z / u) sqrtm(Sigma), kernel by kernel.

The entry points of csrc/mvt.cu are called through the C ABI with (w, V) from numpy's eigh of the same Sigma, so the
package's kernels are measured and cuSOLVER is not.  GEMM-only outputs (Sigma, P, theta) are checked element by
element against a long-double reference with the componentwise bound c (K + 3) u (|A| |B|); the sample, cotangent and
log density against the oracle's formulas written for a given (w, V); the objective value and the three parts of the
gradient (mu, diagonal of F, strict lower triangle of F) norm-wise at 1e-10.  Outputs, gradient and workspace are
filled with NaN before every call.  Then C4 at full size against the oracle, and both eigh fallbacks of
MultivariateT._eigh.
"""
import math
from collections import defaultdict

import numpy as np
import pytest
import torch
from scipy import special as sps

from conftest import relerr
from _problems import hier_problem

pytestmark = pytest.mark.gpu

TOL64 = 1e-10
U = 2.0 ** -53
LD = np.longdouble
ERRS = defaultdict(float)            # largest error seen per group, printed at the end of the module


def _note(key, value):
    ERRS[key] = max(ERRS[key], float(value))


@pytest.fixture(scope='module', autouse=True)
def _report():
    yield
    for k in sorted(ERRS):
        print('[mvt sqrtm] %-40s %.3g' % (k, ERRS[k]))


@pytest.fixture(scope='module')
def vb():
    import viabel_b200
    return viabel_b200


@pytest.fixture(scope='module')
def vo():
    from oracle import viabel_oracle
    return viabel_oracle


def _dev(a):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float64, device='cuda')


def _nan(*shape):
    return torch.full(shape, float('nan'), dtype=torch.float64, device='cuda')


def _nan_ws(nbytes):
    return torch.full((max(int(nbytes), 1),), 255, dtype=torch.uint8, device='cuda')     # all-ones bytes: NaN doubles


def _componentwise(key, out, ref, absprod, K):
    """|out - ref| <= 2 (K + 3) u (|A| |B|) elementwise; records the largest ratio |out - ref| / ((K + 3) u |A| |B|)."""
    err = np.abs(np.asarray(out, dtype=LD) - ref)
    scale = (K + 3) * LD(U) * absprod
    bad = err > 2 * scale
    assert not bad.any(), (key, int(bad.sum()), float(np.max(err - 2 * scale)))
    with np.errstate(divide='ignore', invalid='ignore'):
        ratio = np.where(scale > 0, err / scale, 0.0)
    _note('gemm bound ratio ' + key, np.max(ratio) if ratio.size else 0.0)


def _random_orthogonal(d, rs):
    Q, R = np.linalg.qr(rs.randn(d, d))
    return Q * np.sign(np.diag(R))


def _spd(d, kappa, rs):
    """V diag(w) V^T with eigenvalues from 1 down to 1 / kappa, or ('repeated') half of them equal."""
    if kappa == 'repeated':
        w = np.concatenate([np.full(d - d // 2, 0.7), np.linspace(0.4, 1.6, d // 2)])
    else:
        w = np.logspace(0.0, -np.log10(kappa), d)
    V = _random_orthogonal(d, rs)
    S = (V * w) @ V.T
    return 0.5 * (S + S.T)


def _logpdf_wv(mu, w, V, x, df):
    """_distributions.py:7-38 (oracle mvt_log_density) with the eigen-decomposition given."""
    d = x.shape[1]
    winv = np.where(np.abs(w) <= 1e-10, 0.0, 1.0 / np.where(w == 0, 1.0, w))
    maha = np.sum(((x - mu) @ V) ** 2 * winv, axis=-1)
    with np.errstate(invalid='ignore', divide='ignore'):
        logdet = np.sum(np.log(w))
    return (sps.gammaln(0.5 * (df + d)) - sps.gammaln(0.5 * df) - 0.5 * d * math.log(math.pi * df)
            - 0.5 * logdet - 0.5 * (df + d) * np.log(1.0 + maha / df))


def _objective_ref(vo, vp, chi2, z, f, G, df, w, V, objective, alpha, lib):
    """oracle exclusive_kl_mvt / alpha_divergence_mvt with fixed f, G and the given (w, V); the entropy is the stable
    sum of log L_ii, which the oracle's det form equals where it does not overflow."""
    S, d = z.shape
    mu, L = vo.mvt_unpack(vp, d)
    zu = z / np.sqrt(chi2 / df)[:, None]
    if objective == lib.OBJ_EXCLUSIVE_KL:
        value = -(np.mean(f) + vo.mvt_entropy_stable(vp, d))
        sv, c = np.ones(S), -1.0 / S
        diag_add = -1.0
    else:
        A = (V * np.sqrt(np.maximum(w, 0.0))) @ V.T
        lw = f - _logpdf_wv(mu, w, V, mu + zu @ A, df)
        m = np.max(lw)
        sv = np.exp(lw - m) ** alpha
        value = np.log(np.mean(sv)) / alpha + m
        c = alpha / S
        diag_add = c * np.sum(sv)
    Fbar = vo._mvt_backprop(c * (zu.T @ (sv[:, None] * G)), L, w, V)
    Fbar[np.diag_indices(d)] += diag_add
    return value, np.concatenate([c * (sv @ G), Fbar[np.tril_indices(d)]])


def _grad_parts(g, d):
    packed = g[d:]
    rows = np.repeat(np.arange(d), np.arange(1, d + 1))
    cols = np.arange(packed.size) - rows * (rows + 1) // 2
    return {'mu': g[:d], 'diag': packed[rows == cols], 'lower': packed[rows > cols]}


def _run_kernels(vb, vo, vp, S, df, rs, key):
    """Every sqrtm entry point at one (var_param, S, df) against its reference.  Returns the device outputs."""
    lib, ptr, st, cl = vb._lib.lib, vb._lib.ptr, vb._lib.stream(), vb._lib
    d = int((math.isqrt(8 * vp.size + 9) - 3) // 2)
    assert d + d * (d + 1) // 2 == vp.size
    mu, L0 = vo.mvt_unpack(vp, d)
    vpd = _dev(vp)
    # unpack
    L, hl = _nan(d, d), _nan(1)
    cl.check(lib.vb_mvt_unpack_f64(ptr(vpd), d, ptr(L), ptr(hl), st))
    Lh = L.cpu().numpy()
    assert np.isfinite(Lh).all() and np.isfinite(hl.item())
    assert not np.triu(Lh, 1).any()
    np.testing.assert_allclose(Lh, L0, rtol=8 * U, atol=0)           # exp on the device and in numpy: 1 ulp each
    Fd = vp[d:][np.arange(d) * (np.arange(d) + 3) // 2]                # packed F_ii
    assert abs(hl.item() - np.sum(Fd)) <= 2 * d * U * np.sum(np.abs(Fd))
    # sigma, with a scale
    scale = df / (df - 2.0)
    Sig = _nan(d, d)
    cl.check(lib.vb_mvt_sigma_f64(ptr(L), d, scale, ptr(Sig), st))
    Ll = Lh.astype(LD)
    _componentwise(key, Sig.cpu().numpy(), LD(scale) * (Ll @ Ll.T), abs(LD(scale)) * (np.abs(Ll) @ np.abs(Ll).T), d)
    # eigen-decomposition of the same Sigma on the host
    Sig0 = Lh @ Lh.T
    w, V = np.linalg.eigh(0.5 * (Sig0 + Sig0.T))
    wd, Vd = _dev(w), _dev(V)
    # transform
    chi2, z = rs.chisquare(df, S), rs.randn(S, d)
    zd, cd = _dev(z), _dev(chi2)
    P, theta, zu2 = _nan(S, d), _nan(S, d), _nan(S)
    ws = _nan_ws(lib.vb_mvt_transform_workspace_bytes(S, d))
    cl.check(lib.vb_mvt_transform_f64(ptr(vpd), ptr(zd), ptr(cd), df, S, d, ptr(wd), ptr(Vd), ptr(P), ptr(theta), ptr(zu2),
                                      ptr(ws), ws.numel(), st))
    Ph, th, z2 = P.cpu().numpy(), theta.cpu().numpy(), zu2.cpu().numpy()
    assert np.isfinite(Ph).all() and np.isfinite(th).all() and np.isfinite(z2).all()
    iu = 1.0 / np.sqrt(chi2.astype(LD) / LD(df))
    zl, Vl = z.astype(LD), V.astype(LD)
    _componentwise(key, Ph, iu[:, None] * (zl @ Vl), np.abs(iu)[:, None] * (np.abs(zl) @ np.abs(Vl)), d)
    sw = np.sqrt(np.maximum(w, 0.0).astype(LD))
    Pl = Ph.astype(LD) * sw
    _componentwise(key, th, mu.astype(LD) + Pl @ Vl.T, np.abs(Pl) @ np.abs(Vl).T + np.abs(mu.astype(LD)), d)
    zu = z / np.sqrt(chi2 / df)[:, None]
    A = (V * np.sqrt(np.maximum(w, 0.0))) @ V.T
    e = relerr(th, mu + zu @ A)
    _note('sample ' + key, e)
    assert e < TOL64
    assert relerr(z2, np.sum(zu * zu, axis=1)) < 1e-13
    # objectives with arbitrary f and G
    f, G = rs.randn(S), rs.randn(S, d)
    fd, Gd = _dev(f), _dev(G)
    wso = torch.empty(lib.vb_mvt_objective_workspace_bytes(S, d), dtype=torch.uint8, device='cuda')
    outs = []
    for objective, alpha in ((cl.OBJ_EXCLUSIVE_KL, 0.0), (cl.OBJ_ALPHA, 0.5), (cl.OBJ_ALPHA, 2.0)):
        out = _nan(1 + vp.size)
        wso.fill_(255)
        cl.check(lib.vb_mvt_objective_f64(ptr(L), ptr(hl), ptr(wd), ptr(Vd), ptr(P), ptr(zu2), ptr(fd), ptr(Gd), S, d, df,
                                          objective, alpha, ptr(out[:1]), ptr(out[1:]), ptr(wso), wso.numel(), st))
        o = out.cpu().numpy()
        assert np.isfinite(o).all()                                    # every packed entry written
        v0, g0 = _objective_ref(vo, vp, chi2, z, f, G, df, w, V, objective, alpha, cl)
        e = relerr(o[0], v0)
        _note('objective value ' + key, e)
        assert e < TOL64, ('value', objective, alpha, e)
        got, ref = _grad_parts(o[1:], d), _grad_parts(g0, d)
        for part in ('mu', 'diag', 'lower'):
            if ref[part].size:
                e = relerr(got[part], ref[part])
                _note('objective grad ' + key, e)
                assert e < TOL64, (part, objective, alpha, e)
        outs.append(out)
    # log density at the draws and at points away from them
    x = np.concatenate([mu + zu @ A, mu + 2.0 * rs.randn(min(S, 50), d)])
    lp, xd = _nan(x.shape[0]), _dev(x)
    wsl = _nan_ws(lib.vb_mvt_log_density_workspace_bytes(x.shape[0], d))
    cl.check(lib.vb_mvt_log_density_f64(ptr(vpd), ptr(wd), ptr(Vd), ptr(xd), x.shape[0], d, df, ptr(lp), ptr(wsl),
                                        wsl.numel(), st))
    lph = lp.cpu().numpy()
    assert np.isfinite(lph).all()
    e = relerr(lph, _logpdf_wv(mu, w, V, x, df))
    _note('log density ' + key, e)
    assert e < TOL64
    return dict(L=L, hl=hl, Sigma=Sig, P=P, theta=theta, zu2=zu2, obj=outs, lp=lp)


@pytest.mark.parametrize('d', [1, 5, 31, 32, 33, 63, 64, 65, 130, 257])
@pytest.mark.parametrize('S', [1, 7, 33, 64, 100, 300])
def test_sqrtm_kernels_ragged(vb, vo, d, S):
    """unpack, sigma, transform, objective (ExclusiveKL, AlphaDivergence 0.5 and 2) and log density through the C ABI at
    partial tiles and K slabs, for df = 2.5, 5 and 100, at a correlated Sigma."""
    rs = np.random.RandomState(7919 * d + S)
    B = 0.4 * rs.randn(d, d) / np.sqrt(d)
    vp = vo.mvt_pack(0.5 * rs.randn(d), 0.8 * np.eye(d) + B @ B.T)
    for df in (2.5, 5.0, 100.0):
        _run_kernels(vb, vo, vp, S, df, rs, 'ragged')


@pytest.mark.parametrize('kappa', [1, 1e4, 1e8, 'repeated'])
@pytest.mark.parametrize('d,S', [(65, 100), (257, 300)])
def test_sqrtm_kernels_conditioning(vb, vo, kappa, d, S):
    """Sigma = V diag(w) V^T with a random orthogonal V and condition number 1, 1e4, 1e8, or a repeated eigenvalue.
    The Sylvester solve divides by sqrt(w_a) + sqrt(w_b), a sum and never a difference of eigenvalues, so neither the
    condition number nor equal eigenvalues should cost accuracy: the tolerance stays 1e-10."""
    rs = np.random.RandomState(d + S + (7 if kappa == 'repeated' else int(np.log10(kappa))))
    vp = vo.mvt_pack(0.5 * rs.randn(d), _spd(d, kappa, rs))
    _run_kernels(vb, vo, vp, S, 5.0, rs, 'kappa=%s' % kappa)


def test_sqrtm_kernels_deterministic(vb, vo):
    """Two runs of every entry point on the same inputs give identical bits."""
    d, S = 130, 300
    rs = np.random.RandomState(5)
    vp = vo.mvt_pack(0.5 * rs.randn(d), _spd(d, 1e3, rs))
    a = _run_kernels(vb, vo, vp, S, 5.0, np.random.RandomState(6), 'ragged')
    b = _run_kernels(vb, vo, vp, S, 5.0, np.random.RandomState(6), 'ragged')
    for k in a:
        for x, y in zip(a[k] if k == 'obj' else [a[k]], b[k] if k == 'obj' else [b[k]]):
            assert torch.equal(x, y), k


@pytest.mark.parametrize('edge', ['above', 'at', 'below', 'zero', 'negative'])
def test_log_density_eigenvalue_floor(vb, edge):
    """The reference gives eigenvalues with |w| <= 1e-10 a zero inverse but keeps them in log w: one eigenvalue one ulp
    above 1e-10, exactly 1e-10, one ulp below, 0 and -1e-12.  Finite values agree to 1e-10; NaN and infinity fall on
    the same rows as the reference's."""
    lib, ptr, st, cl = vb._lib.lib, vb._lib.ptr, vb._lib.stream(), vb._lib
    d, n, df = 6, 40, 5.0
    rs = np.random.RandomState(11)
    V = _random_orthogonal(d, rs)
    edge_w = {'above': np.nextafter(1e-10, 1.0), 'at': 1e-10, 'below': np.nextafter(1e-10, 0.0), 'zero': 0.0,
              'negative': -1e-12}[edge]
    w = np.array([2.0, 1.0, 0.5, edge_w, 0.3, 1.5])
    mu = rs.randn(d)
    vp = np.concatenate([mu, np.zeros(d * (d + 1) // 2)])             # only mu is read
    x = mu + rs.randn(n, d)
    x[0] = mu                                                          # the mode: zero Mahalanobis term
    out = _nan(n)
    ws = _nan_ws(lib.vb_mvt_log_density_workspace_bytes(n, d))
    vpd, wd, Vd, xd = _dev(vp), _dev(w), _dev(V), _dev(x)            # held: a freed temporary's memory is reused at once
    cl.check(lib.vb_mvt_log_density_f64(ptr(vpd), ptr(wd), ptr(Vd), ptr(xd), n, d, df, ptr(out), ptr(ws), ws.numel(), st))
    got, ref = out.cpu().numpy(), _logpdf_wv(mu, w, V, x, df)
    np.testing.assert_array_equal(np.isnan(got), np.isnan(ref))
    np.testing.assert_array_equal(np.isinf(got), np.isinf(ref))
    np.testing.assert_array_equal(got[np.isinf(got)], ref[np.isinf(ref)])
    fin = np.isfinite(ref)
    if fin.any():
        assert relerr(got[fin], ref[fin]) < TOL64
    if edge == 'negative':
        assert np.isnan(ref).all()
    elif edge == 'zero':
        assert np.isposinf(ref).all()
    else:
        assert fin.all()


# ---- C4 at full size ------------------------------------------------------------------------------------------------
def _hier_oracle(vo, hp, chunk=32):
    def om(theta):
        parts = [vo.hier_linear_logp_grad(theta[i:i + chunk], hp['X'], hp['y'], hp['group'], hp['G'], hp['p'])
                 for i in range(0, theta.shape[0], chunk)]
        return np.concatenate([a for a, _ in parts]), np.concatenate([b for _, b in parts])
    return om


def _compare_objective(key, d, v, gr, v0, g0):
    v, gr = float(v), gr.cpu().numpy() if torch.is_tensor(gr) else np.asarray(gr)
    e = relerr(v, v0)
    _note(key + ' value', e)
    assert e < TOL64, ('value', e)
    got, ref = _grad_parts(gr, d), _grad_parts(g0, d)
    for part in ('mu', 'diag', 'lower'):
        e = relerr(got[part], ref[part])
        _note(key + ' grad', e)
        assert e < TOL64, (part, e)


@pytest.mark.parametrize('point', ['correlated', 'init'])
def test_sqrtm_c4_full_size_vs_oracle(vb, vo, point):
    """BASELINE configs[3] (d = 2048, S = 256) in the default sqrtm mode, ExclusiveKL and AlphaDivergence(2), against
    the oracle at a correlated point with 2048 distinct eigenvalues in [0.5, 2] and at the reference's init point
    Sigma = 10 I (where cuSOLVER may refuse the matrix and the sort fallback runs).  At Sigma = 10 I the oracle's
    entropy, 0.5 log det(Sigma), overflows (det = 1e2048), so the reference value there uses the same entropy as
    sum log L_ii (mvt_entropy_stable); the gradient needs no change."""
    hp = hier_problem(G=65, p=31, n_per=200, seed=20260118)
    model = vb.HierarchicalLinearRegression(hp['X'], hp['y'], hp['group'], 65)
    d, S = model.dim, 256
    assert d == 2048
    approx = vb.MultivariateT(d, 100)
    rs = np.random.RandomState(2048)
    if point == 'correlated':
        V = _random_orthogonal(d, rs)
        Sigma = (V * rs.permutation(np.linspace(0.5, 2.0, d))) @ V.T
        mu = 0.1 * rs.randn(d)
        mu[d - 2:] = [-1.0, -1.2]
        vp = vo.mvt_pack(mu, 0.5 * (Sigma + Sigma.T))
    else:
        vp = approx.init_param()
    chi2, z = rs.chisquare(100, S), rs.randn(S, d)
    om = _hier_oracle(vo, hp)
    v, gr = vb.ExclusiveKL(approx, model, S)(vp, base=(chi2, z))
    _, g0, f0 = vo.exclusive_kl_mvt(vp, chi2, z, om, 100.0)
    v0 = -(np.mean(f0) + vo.mvt_entropy_stable(vp, d))
    _compare_objective('c4 sqrtm ' + point, d, v, gr, v0, g0)
    v, gr = vb.AlphaDivergence(approx, model, S, 2.0)(vp, base=(chi2, z))
    v0, g0, _ = vo.alpha_divergence_mvt(vp, chi2, z, om, 100.0, 2.0)
    _compare_objective('c4 sqrtm ' + point, d, v, gr, v0, g0)


# ---- eigh fallbacks -------------------------------------------------------------------------------------------------
def _failing_eigh(monkeypatch):
    """torch.linalg.eigh that raises LinAlgError on the first call after each reset of state['calls']."""
    real = torch.linalg.eigh
    state = {'calls': 0}

    def eigh(A, *args, **kwargs):
        state['calls'] += 1
        if state['calls'] == 1:
            raise torch.linalg.LinAlgError('refused (test)')
        return real(A, *args, **kwargs)
    monkeypatch.setattr(torch.linalg, 'eigh', eigh)
    return state


@pytest.mark.parametrize('case', ['ramp-82', 'ramp-250', 'sort-tied', 'sort-distinct'])
def test_eigh_fallbacks_vs_oracle(vb, vo, monkeypatch, case):
    """When cuSOLVER refuses Sigma, MultivariateT._eigh decomposes an exactly diagonal Sigma by sorting its diagonal
    and anything else after adding a relative 1e-13 ramp to the diagonal.  In both branches sample, log_density,
    ExclusiveKL and AlphaDivergence(2) still match the oracle (which decomposes the unperturbed Sigma) to 1e-10."""
    branch, shape = case.split('-')
    G, p, n_per, S = (3, 20, 30, 24) if shape != '250' else (7, 31, 40, 40)
    hp = hier_problem(G=G, p=p, n_per=n_per, seed=31 + G)
    model = vb.HierarchicalLinearRegression(hp['X'], hp['y'], hp['group'], G)
    d = model.dim
    rs = np.random.RandomState(d + len(case))
    if branch == 'ramp':
        B = 0.3 * rs.randn(d, d) / np.sqrt(d)
        Sigma = 0.9 * np.eye(d) + B @ B.T
    elif shape == 'tied':
        Sigma = np.diag(rs.choice([0.5, 1.0, 2.0], d))
    else:
        Sigma = np.diag(rs.permutation(np.linspace(0.5, 2.0, d)))
    vp = vo.mvt_pack(0.2 * rs.randn(d), Sigma)
    calls = 2 if branch == 'ramp' else 1                     # eigh calls per decomposition: refused + ramped, or refused
    state = _failing_eigh(monkeypatch)
    om = lambda th: vo.hier_linear_logp_grad(th, hp['X'], hp['y'], hp['group'], G, p)
    approx = vb.MultivariateT(d, 100)
    chi2, z = rs.chisquare(100, S), rs.randn(S, d)
    key = 'eigh fallback ' + branch
    x = approx.sample(vp, S, base=(chi2, z))
    assert state['calls'] == calls
    x0 = vo.mvt_sample(vp, chi2, z, 100.0)
    e = relerr(x, x0)
    _note(key + ' sample', e)
    assert e < TOL64
    state['calls'] = 0
    lp = approx.log_density(vp, x0)
    assert state['calls'] == calls
    e = relerr(lp, vo.mvt_log_density(vp, x0, 100.0))
    _note(key + ' log density', e)
    assert e < TOL64
    state['calls'] = 0
    v, gr = vb.ExclusiveKL(approx, model, S)(vp, base=(chi2, z))
    assert state['calls'] == calls
    v0, g0, _ = vo.exclusive_kl_mvt(vp, chi2, z, om, 100.0)
    _compare_objective(key, d, v, gr, v0, g0)
    state['calls'] = 0
    v, gr = vb.AlphaDivergence(approx, model, S, 2.0)(vp, base=(chi2, z))
    assert state['calls'] == calls
    v0, g0, _ = vo.alpha_divergence_mvt(vp, chi2, z, om, 100.0, 2.0)
    _compare_objective(key, d, v, gr, v0, g0)
