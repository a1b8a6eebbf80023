"""GPU: the path-derivative ExclusiveKL (use_path_deriv=True) of the full-rank MultivariateT in both
reparameterisations, against the numpy references of tests/_mvt_path_ref.py.

Kernel level through the C ABI with arbitrary f and G: the Cholesky mode at every 64-column block edge (value and the
three parts of the gradient -- mu, diagonal of F, strict lower triangle of F -- norm-wise at 1e-10, outputs and
workspace filled with NaN first, three calls bitwise equal), its on-device solve y = L^-T zhat element by element
against a long-double solve under a first-order bound, and the sqrtm mode with (w, V) from numpy, eigenvalues below
the 1e-10 floor included.  Then the public API on the hierarchical plugin up to C4's full size, sticking the landing
(target = q), unbiasedness, no host synchronisation, convergence, and the C ABI's error returns.
"""
import math
from collections import defaultdict

import numpy as np
import pytest
import torch

import _mvt_path_ref as pr
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
        print('[mvt path] %-44s %.3g' % (k, ERRS[k]))


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


def _grad_parts(g, d):
    packed = g[d:]
    rows = np.repeat(np.arange(d), np.arange(1, d + 1))
    cols = np.arange(packed.size) - rows * (rows + 1) // 2
    return {'mu': g[:d], 'diag': packed[rows == cols], 'lower': packed[rows > cols]}


def _compare(key, d, v, gr, v0, g0):
    v = float(v)
    gr = gr.cpu().numpy() if torch.is_tensor(gr) else np.asarray(gr)
    e = relerr(v, v0)
    _note(key + ' value', e)
    assert e < TOL64, ('value', e)
    got, ref = _grad_parts(gr, d), _grad_parts(g0, d)
    for part in ('mu', 'diag', 'lower'):
        if ref[part].size:
            e = relerr(got[part], ref[part])
            _note(key + ' grad', e)
            assert e < TOL64, (part, e)


def _chol_point(d, rs):
    """Lower-triangular F with off-diagonal entries of size 0.5 / sqrt(d) and diag(L) = exp(0.3 N(0, 1))."""
    F = np.tril(0.5 * rs.randn(d, d) / np.sqrt(d), -1) + np.diag(0.3 * rs.randn(d))
    return np.concatenate([rs.randn(d), F[np.tril_indices(d)]])


def _chol_call(vb, vpd, zd, inv_u, zu2, fd, Gd, S, d, df, objective=None, ws=None, out=None):
    lib, ptr, cl = vb._lib.lib, vb._lib.ptr, vb._lib
    objective = cl.OBJ_EXCLUSIVE_KL_PATH if objective is None else objective
    if ws is None:
        ws = _nan_ws(lib.vb_mvt_chol_path_workspace_bytes(S, d))
    if out is None:
        out = _nan(1 + d + d * (d + 1) // 2)
    rc = lib.vb_mvt_chol_objective_f64(ptr(vpd), ptr(zd), ptr(inv_u), ptr(zu2), ptr(fd), ptr(Gd), S, d, df, objective, 0.0,
                                       ptr(out[:1]), ptr(out[1:]), ptr(ws), ws.numel(), vb._lib.stream())
    return rc, out


def _chol_transform(vb, vpd, zd, cd, S, d, df):
    lib, ptr = vb._lib.lib, vb._lib.ptr
    theta, inv_u, zu2 = _nan(S, d), _nan(S), _nan(S)
    vb._lib.check(lib.vb_mvt_chol_transform_f64(ptr(vpd), ptr(zd), ptr(cd), df, S, d, ptr(theta), ptr(inv_u), ptr(zu2),
                                                vb._lib.stream()))
    return theta, inv_u, zu2


# ---- Cholesky mode, kernel level ------------------------------------------------------------------------------------
@pytest.mark.parametrize('d,S', [(1, 1), (1, 7), (5, 7), (63, 64), (64, 100), (65, 1), (65, 256), (127, 7), (128, 64),
                                 (129, 100), (257, 64), (257, 256), (1000, 7), (1000, 256), (2048, 256)])
def test_cholesky_path_kernels_ragged(vb, vo, d, S):
    """vb_mvt_chol_objective_f64(objective=1) with arbitrary f and G against exclusive_kl_mvt_path_cholesky; NaN in
    outputs and workspace beforehand, every packed entry written; three calls bitwise equal."""
    rs = np.random.RandomState(4099 * d + S)
    df = 5.0
    vp = _chol_point(d, rs)
    chi2, z = rs.chisquare(df, S), rs.randn(S, d)
    f, G = rs.randn(S), rs.randn(S, d)
    vpd, zd, cd, fd, Gd = _dev(vp), _dev(z), _dev(chi2), _dev(f), _dev(G)
    _, inv_u, zu2 = _chol_transform(vb, vpd, zd, cd, S, d, df)
    outs = []
    for _ in range(3):
        rc, out = _chol_call(vb, vpd, zd, inv_u, zu2, fd, Gd, S, d, df)
        vb._lib.check(rc)
        outs.append(out)
    o = outs[0].cpu().numpy()
    assert np.isfinite(o).all()                               # every packed entry written
    v0, g0, _ = pr.exclusive_kl_mvt_path_cholesky(vp, chi2, z, lambda th: (f, G), df)
    _compare('cholesky kernels', d, o[0], o[1:], v0, g0)
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])


def _ld_solve_rows(L, Z):
    """Rows y_s = L^-T z_s in long double by back substitution (L^T y = z)."""
    Lt = L.astype(LD)
    Y = np.zeros(Z.shape, dtype=LD)
    Zl = Z.astype(LD)
    for i in range(L.shape[0] - 1, -1, -1):
        Y[:, i] = (Zl[:, i] - Y[:, i + 1:] @ Lt[i + 1:, i]) / Lt[i, i]
    return Y


@pytest.mark.parametrize('cond', [1.0, 1e2, 1e4, 1e6])
@pytest.mark.parametrize('d', [129, 1000])
def test_cholesky_path_solve_elementwise(vb, vo, cond, d):
    """The on-device y = L^-T zhat (L^-1 by diagonal-block substitution and doubling, then Zhat L^-1), read through
    the mean gradient of a one-draw call with G = 0: grad_mu = -kappa y.  Against a long-double back substitution,
    element by element, under the first-order bound

        |err| <= c d u kappa (|zhat|^T |X| + |zhat|^T |X| |L| |X|),   X = L^-1,  c = 2,

    for L = chol(V diag(w) V^T) with cond(L) = 1 ... 1e6.  The largest err / (d u kappa (...)) is reported."""
    rs = np.random.RandomState(d + int(math.log10(cond)))
    Q, R = np.linalg.qr(rs.randn(d, d))
    V = Q * np.sign(np.diag(R))
    w = np.logspace(0.0, -2.0 * math.log10(cond), d)
    Sig = (V * w) @ V.T
    vp = vo.mvt_pack(rs.randn(d), 0.5 * (Sig + Sig.T))
    _, L = vo.mvt_unpack(vp, d)
    X = np.linalg.inv(L)
    absXLX = np.abs(X) @ (np.abs(L) @ np.abs(X))
    df, n = 5.0, 4
    vpd = _dev(vp)
    worst = 0.0
    for s in range(n):
        chi2, z = rs.chisquare(df, 1), rs.randn(1, d)
        zd, cd = _dev(z), _dev(chi2)
        _, inv_u, zu2 = _chol_transform(vb, vpd, zd, cd, 1, d, df)
        rc, out = _chol_call(vb, vpd, zd, inv_u, zu2, _dev(np.zeros(1)), _dev(np.zeros((1, d))), 1, d, df)
        vb._lib.check(rc)
        gmu = out[1:1 + d].cpu().numpy()
        zu = z.astype(LD) / np.sqrt(chi2.astype(LD) / LD(df))[:, None]
        kappa = (LD(df) + d) / (LD(df) + np.sum(zu * zu))
        ref = -kappa * _ld_solve_rows(L, zu)[0]
        za = np.abs(zu[0]).astype(np.float64)
        scale = d * U * float(kappa) * (za @ np.abs(X) + za @ absXLX)
        err = np.abs(gmu.astype(LD) - ref).astype(np.float64)
        assert (err <= 2.0 * scale).all(), (s, float(np.max(err / scale)))
        worst = max(worst, float(np.max(err / scale)))
    _note('solve err/(d u bound) cond=%g' % cond, worst)


def test_cholesky_path_deterministic_across_workspaces(vb, vo):
    """Different workspace contents (NaN or zeros) and a fresh allocation give identical bits at C4's size."""
    d, S, df = 2048, 256, 100.0
    rs = np.random.RandomState(77)
    vp = _chol_point(d, rs)
    chi2, z = rs.chisquare(df, S), rs.randn(S, d)
    f, G = rs.randn(S), rs.randn(S, d)
    vpd, zd, cd, fd, Gd = _dev(vp), _dev(z), _dev(chi2), _dev(f), _dev(G)
    _, inv_u, zu2 = _chol_transform(vb, vpd, zd, cd, S, d, df)
    nbytes = vb._lib.lib.vb_mvt_chol_path_workspace_bytes(S, d)
    outs = [_chol_call(vb, vpd, zd, inv_u, zu2, fd, Gd, S, d, df, ws=ws)[1]
            for ws in (_nan_ws(nbytes), torch.zeros(nbytes, dtype=torch.uint8, device='cuda'), None)]
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])


# ---- sqrtm mode, kernel level ---------------------------------------------------------------------------------------
def _sqrtm_path_call(vb, vo, vp, S, df, rs, w=None, V=None):
    """unpack -> transform -> vb_mvt_objective_f64(objective=1) with (w, V) from numpy.  Returns (out, ref inputs)."""
    lib, ptr, st, cl = vb._lib.lib, vb._lib.ptr, vb._lib.stream(), vb._lib
    d = int((math.isqrt(8 * vp.size + 9) - 3) // 2)
    vpd = _dev(vp)
    L, hl = _nan(d, d), _nan(1)
    cl.check(lib.vb_mvt_unpack_f64(ptr(vpd), d, ptr(L), ptr(hl), st))
    Lh = L.cpu().numpy()
    if w is None:
        Sig0 = Lh @ Lh.T
        w, V = np.linalg.eigh(0.5 * (Sig0 + Sig0.T))
    wd, Vd = _dev(w), _dev(V)
    chi2, z = rs.chisquare(df, S), rs.randn(S, d)
    zd, cd = _dev(z), _dev(chi2)
    P, theta, zu2 = _nan(S, d), _nan(S, d), _nan(S)
    ws = _nan_ws(lib.vb_mvt_transform_workspace_bytes(S, d))
    cl.check(lib.vb_mvt_transform_f64(ptr(vpd), ptr(zd), ptr(cd), df, S, d, ptr(wd), ptr(Vd), ptr(P), ptr(theta), ptr(zu2),
                                      ptr(ws), ws.numel(), st))
    f, G = rs.randn(S), rs.randn(S, d)
    fd, Gd = _dev(f), _dev(G)
    wso = _nan_ws(lib.vb_mvt_path_workspace_bytes(S, d))
    out = _nan(1 + vp.size)
    cl.check(lib.vb_mvt_objective_f64(ptr(L), ptr(hl), ptr(wd), ptr(Vd), ptr(P), ptr(zu2), ptr(fd), ptr(Gd), S, d, df,
                                      cl.OBJ_EXCLUSIVE_KL_PATH, 0.0, ptr(out[:1]), ptr(out[1:]), ptr(wso), wso.numel(), st))
    return out, (chi2, z, f, G, w, V, float(hl.item()))


@pytest.mark.parametrize('d,S', [(1, 1), (5, 7), (31, 33), (32, 300), (33, 1), (64, 64), (65, 100), (130, 300),
                                 (257, 100)])
def test_sqrtm_path_kernels_ragged(vb, vo, d, S):
    """vb_mvt_objective_f64(objective=1) at partial tiles and K slabs against exclusive_kl_mvt_path with the same
    (w, V); NaN in outputs and workspace beforehand; two calls bitwise equal."""
    rs = np.random.RandomState(7919 * d + S + 1)
    B = 0.4 * rs.randn(d, d) / np.sqrt(d)
    vp = vo.mvt_pack(0.5 * rs.randn(d), 0.8 * np.eye(d) + B @ B.T)
    for df in (2.5, 100.0):
        out, (chi2, z, f, G, w, V, _) = _sqrtm_path_call(vb, vo, vp, S, df, np.random.RandomState(S))
        again, _ = _sqrtm_path_call(vb, vo, vp, S, df, np.random.RandomState(S))
        assert torch.equal(out, again)
        o = out.cpu().numpy()
        assert np.isfinite(o).all()
        v0, g0, _ = pr.exclusive_kl_mvt_path(vp, chi2, z, lambda th: (f, G), df, w=w, V=V)
        _compare('sqrtm kernels', d, o[0], o[1:], v0, g0)


@pytest.mark.parametrize('d,S', [(6, 7), (65, 100), (257, 64)])
def test_sqrtm_path_eigenvalue_floor(vb, vo, d, S):
    """Sigma with eigenvalues 1e-12 (below the reference's 1e-10 floor: zero inverse) and 2e-10 (above it) among
    [0.5, 2]; device and oracle get the same (w, V).

    The value is compared with the oracle's log-determinant 0.5 sum log w swapped for the device's sum_i F_ii: eigh's
    absolute error of about u |Sigma| in an eigenvalue near 1e-12 moves log w by about 1e-4, which is not the device's
    to match.  The gradient: y_s carries 1 / sqrt(2e-10) = 7e4 in the unfloored small direction and the sqrtm VJP
    divides by sqrt(w_a) + sqrt(w_b) >= 2e-6, so a float64 evaluation of the oracle itself is off by up to 2e-10 from
    the same formula in long double at d = 257.  Each part is compared with the long-double evaluation at
    max(1e-10, 4 x the float64 oracle's own error there)."""
    rs = np.random.RandomState(d + S)
    Q, R = np.linalg.qr(rs.randn(d, d))
    Vs = Q * np.sign(np.diag(R))
    ws = rs.uniform(0.5, 2.0, d)
    ws[:2] = [1e-12, 2e-10]
    Sig = (Vs * ws) @ Vs.T
    vp = vo.mvt_pack(0.3 * rs.randn(d), 0.5 * (Sig + Sig.T))
    out, (chi2, z, f, G, w, V, hl) = _sqrtm_path_call(vb, vo, vp, S, 7.0, rs)
    assert np.sum(np.abs(w) <= 1e-10) == 1 and np.sum((w > 1e-10) & (w < 1e-9)) == 1
    o = out.cpu().numpy()
    assert np.isfinite(o).all()
    model = lambda th: (f, G)
    v0, g0, _ = pr.exclusive_kl_mvt_path(vp, chi2, z, model, 7.0, w=w, V=V, half_logdet=hl)
    _, gl, _ = pr.exclusive_kl_mvt_path(vp, chi2.astype(LD), z.astype(LD), model, 7.0, w=w.astype(LD), V=V.astype(LD),
                                        half_logdet=hl)
    e = relerr(o[0], v0)
    _note('sqrtm floor value', e)
    assert e < TOL64
    got, ref, f64 = _grad_parts(o[1:], d), _grad_parts(gl.astype(np.float64), d), _grad_parts(g0, d)
    for part in ('mu', 'diag', 'lower'):
        e, e64 = relerr(got[part], ref[part]), relerr(f64[part], ref[part])
        _note('sqrtm floor grad vs long double', e)
        _note('sqrtm floor grad, float64 oracle vs long double', e64)
        assert e <= max(TOL64, 4.0 * e64), (part, e, e64)


# ---- through the public API -----------------------------------------------------------------------------------------
def _hier_oracle(vo, hp, chunk=32):
    def om(theta):
        parts = [vo.hier_linear_logp_grad(theta[i:i + chunk], hp['X'], hp['y'], hp['group'], hp['G'], hp['p'])
                 for i in range(0, theta.shape[0], chunk)]
        return np.concatenate([a for a, _ in parts]), np.concatenate([b for _, b in parts])
    return om


@pytest.mark.parametrize('reparam', ['sqrtm', 'cholesky'])
@pytest.mark.parametrize('G,p,n_per,S', [(1, 5, 40, 9), (3, 20, 30, 24), (7, 31, 40, 40)])
def test_path_hier_vs_reference(vb, vo, reparam, G, p, n_per, S):
    """ExclusiveKL(MultivariateT(d, 100[, reparam]), model, S, use_path_deriv=True) on the hierarchical plugin at
    d = 12, 82, 250."""
    hp = hier_problem(G=G, p=p, n_per=n_per, seed=31 + G)
    model = vb.HierarchicalLinearRegression(hp['X'], hp['y'], hp['group'], G)
    d = model.dim
    rs = np.random.RandomState(d)
    B = 0.3 * rs.randn(d, d) / np.sqrt(d)
    vp = vo.mvt_pack(0.2 * rs.randn(d), 0.9 * np.eye(d) + B @ B.T)
    chi2, z = rs.chisquare(100, S), rs.randn(S, d)
    approx = vb.MultivariateT(d, 100, reparam=reparam)
    v, gr = vb.ExclusiveKL(approx, model, S, use_path_deriv=True)(vp, base=(chi2, z))
    ref = pr.exclusive_kl_mvt_path if reparam == 'sqrtm' else pr.exclusive_kl_mvt_path_cholesky
    v0, g0, _ = ref(vp, chi2, z, _hier_oracle(vo, hp), 100.0)
    _compare('hier %s d=%d' % (reparam, d), d, v, gr, v0, g0)


def test_path_c4_full_size_cholesky(vb, vo):
    """C4 (d = 2048, S = 256) in the Cholesky mode at the point of test_cholesky_c4_full_size_vs_oracle."""
    hp = hier_problem(G=65, p=31, n_per=200, seed=20260118)
    model = vb.HierarchicalLinearRegression(hp['X'], hp['y'], hp['group'], 65)
    d, S = model.dim, 256
    assert d == 2048
    rs = np.random.RandomState(4)
    F = np.tril(0.002 * rs.randn(d, d), -1) + np.diag(0.5 * np.log(0.01) + 0.05 * rs.randn(d))
    vp = np.concatenate([0.1 * rs.randn(d), F[np.tril_indices(d)]])
    vp[d - 2:d] = [-1.0, -1.2]
    chi2, z = rs.chisquare(100, S), rs.randn(S, d)
    approx = vb.MultivariateT(d, 100, reparam='cholesky')
    v, gr = vb.ExclusiveKL(approx, model, S, use_path_deriv=True)(vp, base=(chi2, z))
    v0, g0, _ = pr.exclusive_kl_mvt_path_cholesky(vp, chi2, z, _hier_oracle(vo, hp), 100.0)
    _compare('c4 cholesky', d, v, gr, v0, g0)


@pytest.mark.parametrize('point', ['correlated', 'init'])
def test_path_c4_full_size_sqrtm(vb, vo, point):
    """C4 (d = 2048, S = 256) in the sqrtm mode at the points of test_sqrtm_c4_full_size_vs_oracle.  The device's
    eigen-decomposition is cuSOLVER's (or its fallback at Sigma = 10 I) and the oracle's numpy's; the path gradient
    depends on Sigma^+ and sqrtm(Sigma) only, so it does not matter which eigenvectors either picks."""
    hp = hier_problem(G=65, p=31, n_per=200, seed=20260118)
    model = vb.HierarchicalLinearRegression(hp['X'], hp['y'], hp['group'], 65)
    d, S = model.dim, 256
    approx = vb.MultivariateT(d, 100)
    rs = np.random.RandomState(2048)
    if point == 'correlated':
        Q, R = np.linalg.qr(rs.randn(d, d))
        V = Q * np.sign(np.diag(R))
        Sigma = (V * rs.permutation(np.linspace(0.5, 2.0, d))) @ V.T
        mu = 0.1 * rs.randn(d)
        mu[d - 2:] = [-1.0, -1.2]
        vp = vo.mvt_pack(mu, 0.5 * (Sigma + Sigma.T))
    else:
        vp = approx.init_param()
    chi2, z = rs.chisquare(100, S), rs.randn(S, d)
    v, gr = vb.ExclusiveKL(approx, model, S, use_path_deriv=True)(vp, base=(chi2, z))
    v0, g0, _ = pr.exclusive_kl_mvt_path(vp, chi2, z, _hier_oracle(vo, hp), 100.0)
    _compare('c4 sqrtm ' + point, d, v, gr, v0, g0)


# ---- as an estimator ------------------------------------------------------------------------------------------------
def _t_model(vb, vp, d, df):
    """The family's own log density at var_param vp as a target, closed form with its gradient."""
    from oracle import viabel_oracle as vo
    mu, L = vo.mvt_unpack(vp, d)
    mut, Lt = torch.as_tensor(mu, device='cuda'), torch.as_tensor(L, device='cuda')
    const = (math.lgamma(0.5 * (df + d)) - math.lgamma(0.5 * df) - 0.5 * d * math.log(math.pi * df)
             - float(np.sum(np.log(np.diag(L)))))

    def parts(theta):
        r = (theta - mut).T
        e = torch.linalg.solve_triangular(Lt, r, upper=False)                  # L^-1 (theta - mu)
        delta = (e * e).sum(dim=0)
        y = torch.linalg.solve_triangular(Lt.T, e, upper=True).T               # Sigma^-1 (theta - mu), rows
        return delta, y

    def logp(theta):
        delta, _ = parts(theta)
        return const - 0.5 * (df + d) * torch.log1p(delta / df)

    def grad(theta):
        delta, y = parts(theta)
        return -((df + d) / (df + delta))[:, None] * y
    return vb.Model(logp, grad)


@pytest.mark.parametrize('reparam', ['sqrtm', 'cholesky'])
@pytest.mark.parametrize('d', [4, 130])
def test_path_sticks_the_landing(vb, vo, reparam, d):
    """Target = q at lambda*: every draw's path gradient is zero, so the estimate vanishes to 1e-10 of the norm of
    either of its terms (the model's G and the score kappa y), while the entropy-form gradient at the same draws does
    not."""
    df, S = 9.0, 64
    rs = np.random.RandomState(d + 5)
    B = 0.5 * rs.randn(d, d) / np.sqrt(d)
    vp = vo.mvt_pack(rs.randn(d), 0.7 * np.eye(d) + B @ B.T)
    model = _t_model(vb, vp, d, df)
    approx = vb.MultivariateT(d, df, reparam=reparam)
    chi2, z = rs.chisquare(df, S), rs.randn(S, d)
    vpd = torch.as_tensor(vp, device='cuda')
    _, g_path = vb.ExclusiveKL(approx, model, S, use_path_deriv=True)(vpd, base=(chi2, z))
    _, g_ent = vb.ExclusiveKL(approx, model, S)(vpd, base=(chi2, z))
    ref = pr.exclusive_kl_mvt_path if reparam == 'sqrtm' else pr.exclusive_kl_mvt_path_cholesky
    zero_g = lambda th: (np.zeros(th.shape[0]), np.zeros_like(th))
    _, score_term, _ = ref(vp, chi2, z, zero_g, df)                  # the kappa y term alone
    theta = approx.sample(vp, S, base=(chi2, z))
    Gm = model.logp_and_grad(torch.as_tensor(theta, device='cuda'))[1].cpu().numpy()
    _, both, _ = ref(vp, chi2, z, lambda th: (np.zeros(th.shape[0]), Gm), df)
    model_term = both - score_term
    g_path = g_path.cpu().numpy()
    ratio = np.linalg.norm(g_path) / min(np.linalg.norm(model_term), np.linalg.norm(score_term))
    _note('landing |g| / |term| %s' % reparam, ratio)
    assert ratio <= 1e-10, ratio
    assert np.linalg.norm(g_ent.cpu().numpy()) > 1e-3 * np.linalg.norm(model_term)


def _gaussian_model(vb, m, P):
    Pt, mt = torch.as_tensor(P, device='cuda'), torch.as_tensor(m, device='cuda')

    def logp(theta):
        r = theta - mt
        return -0.5 * ((r @ Pt) * r).sum(dim=1)
    return vb.Model(logp, lambda theta: -(theta - mt) @ Pt)


@pytest.mark.parametrize('reparam', ['sqrtm', 'cholesky'])
def test_path_gradient_unbiased(vb, vo, reparam):
    """The target of test_exclusive_kl_gradient_unbiased: the score term has mean zero, so the path estimator has the
    entropy form's expectation, closed form.  The mean of 400 path gradients lies within 5 standard errors of it."""
    d, df, S, n = 4, 8.0, 16, 400
    rs = np.random.RandomState(3)
    B = rs.randn(d, d) / np.sqrt(d)
    P = np.eye(d) + B @ B.T
    m = rs.randn(d)
    Bq = 0.8 * rs.randn(d, d) / np.sqrt(d)
    vp = vo.mvt_pack(0.2 * rs.randn(d), 0.6 * np.eye(d) + Bq @ Bq.T)
    mu, L = vo.mvt_unpack(vp, d)
    k = df / (df - 2.0)
    Fbar = np.tril(k * P @ L)
    Fbar[np.diag_indices(d)] = Fbar[np.diag_indices(d)] * np.diag(L) - 1.0
    g_true = np.concatenate([P @ (mu - m), Fbar[np.tril_indices(d)]])
    approx = vb.MultivariateT(d, df, seed=21, reparam=reparam)
    obj = vb.ExclusiveKL(approx, _gaussian_model(vb, m, P), S, use_path_deriv=True)
    vpd = torch.as_tensor(vp, device='cuda')
    grads = torch.stack([obj(vpd)[1] for _ in range(n)]).cpu().numpy()
    se = grads.std(axis=0, ddof=1) / np.sqrt(n)
    assert (se > 0).all()
    assert np.max(np.abs(grads.mean(axis=0) - g_true) / se) < 5.0


def test_cholesky_path_no_host_sync(vb, vo):
    """An evaluation plus an RMSProp step with a device var_param enqueues no host synchronisation."""
    hp = hier_problem(G=7, p=31, n_per=40, seed=38)
    model = vb.HierarchicalLinearRegression(hp['X'], hp['y'], hp['group'], 7)
    d, S = model.dim, 100
    rs = np.random.RandomState(9)
    B = 0.3 * rs.randn(d, d) / np.sqrt(d)
    vp = torch.as_tensor(vo.mvt_pack(0.2 * rs.randn(d), 0.9 * np.eye(d) + B @ B.T), device='cuda')
    approx = vb.MultivariateT(d, 100, reparam='cholesky')
    obj = vb.ExclusiveKL(approx, model, S, use_path_deriv=True)
    opt = vb.RMSProp(1e-3)
    obj(vp)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode('error')
    try:
        for _ in range(2):
            _, g = obj(vp)
            opt._fused_step(vp, g, False)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert bool(torch.isfinite(vp).all())


@pytest.mark.parametrize('reparam', ['sqrtm', 'cholesky'])
def test_path_rmsprop_converges(vb, reparam):
    """RMSProp with the path estimator recovers a correlated 3-D Gaussian's mean and covariance to 0.05."""
    m = np.array([1.0, -2.0, 0.5])
    C = np.array([[1.0, 0.5, 0.2], [0.5, 2.0, -0.3], [0.2, -0.3, 0.5]])
    np.random.seed(0)
    approx = vb.MultivariateT(3, 100, seed=2, reparam=reparam)
    obj = vb.ExclusiveKL(approx, _gaussian_model(vb, m, np.linalg.inv(C)), 50, use_path_deriv=True)
    res = vb.RMSProp(0.01).optimize(4000, obj, approx.init_param())
    mean, cov = approx.mean_and_cov(res['opt_param'])
    assert np.max(np.abs(mean - m)) < 0.05, mean
    assert np.max(np.abs(cov - C)) < 0.05, cov


# ---- C ABI errors ---------------------------------------------------------------------------------------------------
def test_path_cabi_errors_write_nothing(vb, vo):
    """Bad arguments, objective 3 and a workspace one byte below the path query each return an error and leave the
    outputs and the workspace untouched, in both modes."""
    lib, ptr, st, cl = vb._lib.lib, vb._lib.ptr, vb._lib.stream(), vb._lib
    d, S, df = 70, 9, 5.0
    rs = np.random.RandomState(1)
    vp = _chol_point(d, rs)
    vpd, zd, cd = _dev(vp), _dev(rs.randn(S, d)), _dev(rs.chisquare(df, S))
    fd, Gd = _dev(rs.randn(S)), _dev(rs.randn(S, d))
    _, inv_u, zu2 = _chol_transform(vb, vpd, zd, cd, S, d, df)
    need = lib.vb_mvt_chol_path_workspace_bytes(S, d)
    assert need > lib.vb_mvt_chol_objective_workspace_bytes(S, d)
    ws = torch.full((need,), 7, dtype=torch.uint8, device='cuda')
    out = torch.full((1 + vp.size,), 3.5, dtype=torch.float64, device='cuda')

    def chol(objective=cl.OBJ_EXCLUSIVE_KL_PATH, nbytes=need, S_=S, z_=zd):
        return lib.vb_mvt_chol_objective_f64(ptr(vpd), ptr(z_), ptr(inv_u), ptr(zu2), ptr(fd), ptr(Gd), S_, d, df, objective,
                                             0.0, ptr(out[:1]), ptr(out[1:]), ptr(ws), nbytes, st)
    assert chol(z_=None) == cl.VB_ERR_INVALID_ARG
    assert chol(S_=0) == cl.VB_ERR_INVALID_ARG
    assert chol(objective=3) == cl.VB_ERR_UNSUPPORTED
    assert chol(nbytes=need - 1) == cl.VB_ERR_WORKSPACE
    torch.cuda.synchronize()
    assert bool((out == 3.5).all()) and bool((ws == 7).all())
    # sqrtm mode
    L, hl = _nan(d, d), _nan(1)
    cl.check(lib.vb_mvt_unpack_f64(ptr(vpd), d, ptr(L), ptr(hl), st))
    Lh = L.cpu().numpy()
    w, V = np.linalg.eigh(Lh @ Lh.T)
    wd, Vd = _dev(w), _dev(V)
    P = _dev(rs.randn(S, d))
    need = lib.vb_mvt_path_workspace_bytes(S, d)
    assert need > lib.vb_mvt_objective_workspace_bytes(S, d)
    ws = torch.full((need,), 7, dtype=torch.uint8, device='cuda')

    def sq(objective=cl.OBJ_EXCLUSIVE_KL_PATH, nbytes=need, S_=S, P_=P):
        return lib.vb_mvt_objective_f64(ptr(L), ptr(hl), ptr(wd), ptr(Vd), ptr(P_), ptr(zu2), ptr(fd), ptr(Gd), S_, d, df,
                                        objective, 0.0, ptr(out[:1]), ptr(out[1:]), ptr(ws), nbytes, st)
    assert sq(P_=None) == cl.VB_ERR_INVALID_ARG
    assert sq(S_=0) == cl.VB_ERR_INVALID_ARG
    assert sq(objective=3) == cl.VB_ERR_UNSUPPORTED
    assert sq(nbytes=need - 1) == cl.VB_ERR_WORKSPACE
    torch.cuda.synchronize()
    assert bool((out == 3.5).all()) and bool((ws == 7).all())
