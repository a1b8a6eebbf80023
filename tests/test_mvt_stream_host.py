"""CPU: the Philox stream layout each family reports through stream_length, which base_draws and streaming
vi_diagnostics advance by: chi-squares first, then normals, each run rounded up to even, for MultivariateT; n d
variates rounded up to even for the mean-field families."""
import pytest


@pytest.mark.parametrize('n,d', [(1, 1), (1, 2), (2, 3), (3, 3), (60011, 7), (100000000, 256)])
def test_stream_length(n, d):
    import viabel_b200 as vb
    nd = n * d
    for reparam in ('sqrtm', 'cholesky'):
        assert vb.MultivariateT(d, 5, reparam=reparam).stream_length(n) == n + (n & 1) + nd + (nd & 1)
    assert vb.MFGaussian(d).stream_length(n) == nd + (nd & 1)
    assert vb.MFStudentT(d, 5).stream_length(n) == nd + (nd & 1)
