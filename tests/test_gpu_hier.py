"""GPU: the hierarchical linear regression plugin (csrc/hier.cu) at its edges -- p = 1, 31 and the largest accepted
p = 32, sample counts around the 128-sample tile, and unequal groups (one empty, one of 130 rows, more than two 64-row
staging passes) given with unsorted labels -- against the oracle's hier_linear_logp_grad at 1e-10."""
import numpy as np
import pytest
import torch

from conftest import relerr

pytestmark = pytest.mark.gpu

TOL64 = 1e-10
SIZES = [3, 0, 130, 1, 64, 17]           # rows per group


@pytest.fixture(scope='module')
def vb():
    import viabel_b200
    return viabel_b200


@pytest.fixture(scope='module')
def vo():
    from oracle import viabel_oracle
    return viabel_oracle


def _problem(p, seed):
    rs = np.random.RandomState(seed)
    group = np.repeat(np.arange(len(SIZES)), SIZES)
    perm = rs.permutation(group.size)
    group = group[perm]                                  # labels in no particular order
    X = rs.randn(group.size, p)
    y = rs.randn(group.size)
    return X, y, group, rs


@pytest.mark.parametrize('p', [1, 31, 32])
@pytest.mark.parametrize('S', [1, 127, 128, 129, 300])
def test_hier_plugin_edges_vs_oracle(vb, vo, p, S):
    X, y, group, rs = _problem(p, 10 * p + S)
    G = len(SIZES)
    model = vb.HierarchicalLinearRegression(X, y, group, G)
    D = model.dim
    assert D == G * p + p + 2
    theta = 0.3 * rs.randn(S, D)
    theta[:, -2:] += [-0.5, 0.2]
    td = torch.as_tensor(theta, device='cuda')
    lp, g = model.logp_and_grad(td)
    lp0, g0 = vo.hier_linear_logp_grad(theta, X, y, group, G, p)
    assert bool(torch.isfinite(lp).all()) and bool(torch.isfinite(g).all())
    assert relerr(lp.cpu().numpy(), lp0) < TOL64
    assert relerr(g.cpu().numpy(), g0) < TOL64
    # the empty group's coefficients see the prior only
    e0 = slice(1 * p, 2 * p)
    assert relerr(g.cpu().numpy()[:, e0], g0[:, e0]) < TOL64
    lp2, none = model.logp_and_grad(td, want_grad=False)
    assert none is None and torch.equal(lp, lp2)


def test_hier_plugin_rejects_p33(vb):
    """p = 33 is refused by the model and by the C ABI (the kernel keeps at most 32 coefficients in registers)."""
    X, y, group, _ = _problem(33, 1)
    with pytest.raises(NotImplementedError):
        vb.HierarchicalLinearRegression(X, y, group, len(SIZES))
    lib = vb._lib.lib
    G, p, S = len(SIZES), 33, 4
    t = lambda a: torch.as_tensor(np.ascontiguousarray(a), device='cuda')
    goff = t(np.concatenate([[0], np.cumsum(SIZES)]).astype(np.int64))
    order = np.argsort(group, kind='stable')
    Xd, yd = t(X[order]), t(y[order])
    theta = torch.zeros(S, G * p + p + 2, dtype=torch.float64, device='cuda')
    lp = torch.empty(S, dtype=torch.float64, device='cuda')
    ws = torch.empty(lib.vb_hier_workspace_bytes(G, S), dtype=torch.uint8, device='cuda')
    rc = lib.vb_hier_logp_grad_f64(Xd.data_ptr(), yd.data_ptr(), goff.data_ptr(), X.shape[0], p, G, theta.data_ptr(), S,
                                   lp.data_ptr(), None, ws.data_ptr(), ws.numel(), vb._lib.stream())
    assert rc == vb._lib.VB_ERR_UNSUPPORTED
