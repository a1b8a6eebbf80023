"""CPU: what the fused AlphaDivergence step rests on.  (1) Drawing the per-step seeds of a chunk of m iterations as one
vectorised np.random.randint call gives the seeds, and leaves the global RNG in the state, of the m scalar draws the
unfused loop makes (objectives.py:455), however the iterations are cut into chunks.  (2) The step's decomposition of
the alpha value and gradient into likelihood sweep sums and per-column prior sums (tests/_alpha_step_ref.py) equals
the oracle, including weights that underflow to zero."""
import numpy as np
import pytest

import _alpha_step_ref as A
from _problems import logistic_problem
from conftest import relerr
from oracle import viabel_oracle as vo


def _same_state(a, b):
    return a[0] == b[0] and np.array_equal(a[1], b[1]) and tuple(a[2:]) == tuple(b[2:])


@pytest.mark.parametrize('chunks', [[1], [7], [100, 100, 50], [3, 1, 999, 2], [1000]])
def test_chunked_seed_draws_equal_scalar_draws(chunks):
    n = sum(chunks)
    np.random.seed(1234)
    np.random.rand(3)                                           # an RNG that is not freshly seeded
    scalar = np.array([np.random.randint(2 ** 32, dtype=np.uint64) for _ in range(n)], dtype=np.uint64)
    after_scalar = np.random.get_state()
    np.random.seed(1234)
    np.random.rand(3)
    parts = [np.random.randint(2 ** 32, dtype=np.uint64, size=m) for m in chunks]
    after_chunks = np.random.get_state()
    assert all(p.dtype == np.uint64 for p in parts)
    assert np.array_equal(np.concatenate(parts), scalar)
    assert _same_state(after_scalar, after_chunks)
    # and the next draw of any kind continues identically
    np.random.set_state(after_scalar)
    a = np.random.randn(5)
    np.random.set_state(after_chunks)
    assert np.array_equal(a, np.random.randn(5))


@pytest.mark.parametrize('family,df', [('gaussian', None), ('student', 6.5)])
@pytest.mark.parametrize('alpha', [0.5, 2.0, 5.0])
@pytest.mark.parametrize('N,d,S', [(200, 7, 1), (300, 13, 7), (150, 33, 100)])
def test_step_decomposition_matches_oracle(family, df, alpha, N, d, S):
    X, y, beta = logistic_problem(N, d, seed=N + d + S)
    rs = np.random.RandomState(S)
    base = rs.randn(S, d) if family == 'gaussian' else rs.standard_t(df, size=(S, d))
    vp = np.concatenate([0.5 * beta, -1.0 + 0.1 * rs.randn(d)])
    v, g, lw = A.alpha_step(vp, base, X, y, 10.0, alpha, family, df)
    v0, g0, lw0 = vo.alpha_divergence_meanfield(vp, base, lambda th: vo.logistic_logp_grad(th, X, y, 10.0), alpha,
                                                family, df)
    assert relerr(lw, lw0) < 1e-13
    assert relerr(v, v0) < 1e-13
    assert relerr(g, g0) < 1e-12


def test_step_decomposition_with_underflowing_weights():
    """log-weights spread over thousands: all but a few weights are exactly zero, and the decomposition still equals
    the oracle (the GPU tests use the same construction)."""
    N, d, S, alpha = 2000, 40, 64, 5.0
    X, y, beta = logistic_problem(N, d, seed=9)
    rs = np.random.RandomState(10)
    base = rs.randn(S, d)
    vp = np.concatenate([beta, 1.5 * np.ones(d)])
    v, g, lw = A.alpha_step(vp, base, X, y, 10.0, alpha)
    v0, g0, lw0 = vo.alpha_divergence_meanfield(vp, base, lambda th: vo.logistic_logp_grad(th, X, y, 10.0), alpha)
    w = np.exp(lw0 - lw0.max()) ** alpha
    assert np.mean(w == 0.0) > 0.5 and lw0.max() - lw0.min() > 1000
    assert relerr(v, v0) < 1e-13 and relerr(g, g0) < 1e-12
