"""CPU: the identity the streamed LRGaussian log-weights rest on (log q from |u|^2 - |P u|^2, no solve per draw),
against the oracle's dense density where that is accurate and against 40-digit mpmath where B dominates sigma; and
the Philox stream layout LRGaussian.stream_length reports (z run, then eps run, each rounded up to even)."""
import numpy as np
import pytest

import _lr_stream_ref as lr


@pytest.fixture(scope='module')
def vo():
    from oracle import viabel_oracle
    return viabel_oracle


@pytest.mark.parametrize('d,k', [(1, 1), (5, 0), (20, 3), (31, 8), (4, 9)])
@pytest.mark.parametrize('ratio', [0.1, 1.0, 10.0])
def test_identity_vs_oracle(vo, d, k, ratio):
    rs = np.random.RandomState(d * 100 + k)
    vp = lr.point(d, k, ratio, rs)
    z, eps = rs.randn(50, k), rs.randn(50, d)
    ref = vo.lr_log_density(vp, vo.lr_sample(vp, z, eps), k)
    got = lr.log_density_from_base(vp, z, eps, lr.projection(vp, d, k))
    assert np.linalg.norm(got - ref) / np.linalg.norm(ref) < 1e-12


@pytest.mark.parametrize('ratio', [1.0, 1e2, 1e4, 1e6])
def test_identity_vs_mpmath(ratio):
    d, k = 20, 3
    rs = np.random.RandomState(int(np.log10(ratio)) + 7)
    vp = lr.point(d, k, ratio, rs)
    z, eps = rs.randn(12, k), rs.randn(12, d)
    ref = lr.mp_log_density(vp, z, eps)
    got = lr.log_density_from_base(vp, z, eps, lr.projection(vp, d, k))
    assert np.linalg.norm(got - ref) / np.linalg.norm(ref) < 1e-10


def test_projection_rows_orthonormal():
    d, k = 12, 4
    P = lr.projection(lr.point(d, k, 3.0, np.random.RandomState(0)), d, k)
    np.testing.assert_allclose(P @ P.T, np.eye(k), atol=1e-13)
    assert np.allclose(np.triu(P[:, :k], 1), 0.0) and np.all(np.diag(P[:, :k]) > 0)


@pytest.mark.parametrize('n,d,k', [(1, 1, 0), (3, 3, 0), (1, 2, 1), (3, 2, 3), (3, 3, 1), (7, 5, 3), (60011, 7, 4),
                                   (100000000, 256, 8), (5000000, 1000, 16)])
def test_stream_length(n, d, k):
    import viabel_b200 as vb
    nk, nd = n * k, n * d
    assert vb.LRGaussian(d, 5, k).stream_length(n) == nk + (nk & 1) + nd + (nd & 1)
