"""GPU: the full-rank kernels at batch sizes past what a launch's gridDim.y (65 535) or 32-bit grid arithmetic would
allow: every such launch numbers its tiles on gridDim.x or strides over rows.  Rows past each old limit are compared
with the oracle, not only norm-wise over the whole batch."""
import numpy as np
import pytest
import torch

import _mvt_cholesky_ref as cr
from conftest import relerr
from _problems import hier_problem

pytestmark = pytest.mark.gpu

TOL64 = 1e-10


@pytest.fixture(scope='module')
def vb():
    import viabel_b200
    return viabel_b200


@pytest.fixture(scope='module')
def vo():
    from oracle import viabel_oracle
    return viabel_oracle


def _point(vo, d, rs):
    B = 0.5 * rs.randn(d, d)
    return vo.mvt_pack(rs.randn(d), 0.5 * np.eye(d) + B @ B.T)


def _check_rows(got, ref, first_new):
    assert np.isfinite(got).all()
    assert relerr(got, ref) < TOL64
    assert relerr(got[first_new:], ref[first_new:]) < TOL64


def test_sqrtm_sample_and_log_density_past_65535_gemm_tiles(vb, vo):
    """n = 4 200 000 draws at d = 3: the S x d x d GEMMs of the transform and the log density have 65 625 row tiles."""
    n, d, df = 4_200_000, 3, 10.0
    rs = np.random.RandomState(3)
    vp = _point(vo, d, rs)
    chi2, z = rs.chisquare(df, n), rs.randn(n, d)
    approx = vb.MultivariateT(d, df)
    x = approx.sample(vp, n, base=(chi2, z))
    x0 = vo.mvt_sample(vp, chi2, z, df)
    _check_rows(x, x0, 65535 * 64)
    _check_rows(approx.log_density(vp, x0), vo.mvt_log_density(vp, x0, df), 65535 * 64)


def test_sqrtm_sample_past_int32_row_arithmetic(vb, vo):
    """n = 2^26 + 1000 draws at d = 1: 32 n no longer fits an int, which the per-sample row kernel's grid once used."""
    n, df = 2 ** 26 + 1000, 10.0
    rs = np.random.RandomState(26)
    vp = np.array([0.3, 0.2])
    chi2, z = rs.chisquare(df, n), rs.randn(n, 1)
    x = vb.MultivariateT(1, df).sample(vp, n, base=(chi2, z))
    _check_rows(x, vo.mvt_sample(vp, chi2, z, df), 2 ** 26 - 8)


def test_cholesky_sample_past_65535_row_tiles(vb, vo):
    """n = 2 200 000 in Cholesky mode: 68 750 tiles of 32 samples."""
    n, d, df = 2_200_000, 3, 10.0
    rs = np.random.RandomState(5)
    vp = _point(vo, d, rs)
    chi2, z = rs.chisquare(df, n), rs.randn(n, d)
    x = vb.MultivariateT(d, df, reparam='cholesky').sample(vp, n, base=(chi2, z))
    _check_rows(x, cr.mvt_sample_cholesky(vp, chi2, z, df), 65535 * 32)


def test_hier_plugin_past_65535_sample_tiles(vb, vo):
    """S = 8 400 000 samples of a one-group model (65 625 tiles of 128 samples): a strided subset of the rows and every
    row past 8 388 480 against the oracle."""
    hp = hier_problem(G=1, p=2, n_per=50, seed=8)
    model = vb.HierarchicalLinearRegression(hp['X'], hp['y'], hp['group'], 1)
    S, D = 8_400_000, model.dim
    gen = torch.Generator(device='cuda').manual_seed(8)
    theta = 0.3 * torch.randn(S, D, dtype=torch.float64, device='cuda', generator=gen)
    lp, g = model.logp_and_grad(theta)
    assert bool(torch.isfinite(lp).all()) and bool(torch.isfinite(g).all())
    rows = np.concatenate([np.arange(0, S, 997), np.arange(65535 * 128, S)])
    idx = torch.as_tensor(rows, device='cuda')
    lp0, g0 = vo.hier_linear_logp_grad(theta[idx].cpu().numpy(), hp['X'], hp['y'], hp['group'], 1, 2)
    assert relerr(lp[idx].cpu().numpy(), lp0) < TOL64
    assert relerr(g[idx].cpu().numpy(), g0) < TOL64
    tail = rows >= 65535 * 128
    assert relerr(lp[idx].cpu().numpy()[tail], lp0[tail]) < TOL64


def test_vi_diagnostics_multivariate_t_5e6(vb, vo):
    """vi_diagnostics of MultivariateT(3, 10) with 5 000 000 draws (kept in memory: 120 MB) runs to the end, and its
    k-hat is the oracle's psislw of the numpy log weights at the same draws."""
    d, df, n = 3, 10.0, 5_000_000
    mean, sd = np.array([0.5, -1.0, 2.0]), np.array([1.0, 0.7, 1.3])
    vp = vo.mvt_pack(mean + 0.05, np.diag((1.1 * sd) ** 2))
    model = vb.GaussianTarget(mean, sd)
    report = vb.vi_diagnostics(vp, model=model, approx=vb.MultivariateT(d, df), n_samples=n)
    assert 'd2' in report and np.isfinite(report['d2'])
    draws = np.asarray(report['samples']).T
    assert draws.shape == (n, d)
    lw = vo.gauss_target_logp_grad(draws, mean, sd)[0] - vo.mvt_log_density(vp, draws, df)
    _, khat0 = vo.psislw(lw)
    assert relerr(report['khat'], khat0) < 1e-9
