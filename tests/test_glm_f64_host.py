"""Host checks of the float64 reference and error model of the exact GLM kernels (tests/_glm_f64_ref.py)."""
import numpy as np
import pytest

from _glm_f64_ref import (CASES, Reference, alpha_weights, case_links, case_seed, detected, link_terms, ll_rtol,
                          make_case, mp_link, mutations, plan)


def test_plan_regimes():
    """The mirror of make_plan: X-tile height and per-warp ge rows by d, for the sweep's 16 warps."""
    want = [(1, 576, 32, True), (577, 832, 32, False), (833, 864, 16, True), (865, 1600, 16, False),
            (1601, 2896, 8, False)]
    for lo, hi, bm, priv in want:
        for d in (lo, hi):
            assert plan(d) == (bm, priv), d
    assert plan(2897) is None


def test_reference_matches_the_oracle():
    """Sign and weight conventions against the oracle's logistic and probit log densities."""
    from oracle import viabel_oracle as vo
    N, d, S = 700, 19, 9
    for link, fn in (('logistic', vo.logistic_logp_grad), ('probit', vo.probit_logp_grad)):
        X, y, theta, base, _ = make_case(N, d, S, link, 5, saturate=False)
        w = alpha_weights(S, 3)
        ref = Reference(X, y, theta, base, link, w=w)
        f, g = fn(theta, X, y, 10.0)
        lp = -0.5 * np.sum(theta ** 2, axis=1) / 100.0 - 0.5 * d * np.log(2 * np.pi * 100.0)
        gl = g + theta / 100.0
        assert np.allclose(ref.ll, f - lp, rtol=1e-12, atol=1e-9)
        assert np.allclose(ref.gmu, w @ gl, rtol=1e-11, atol=1e-9)
        assert np.allclose(ref.ge, np.sum(w[:, None] * gl * base, axis=0), rtol=1e-11, atol=1e-9)


def test_gaussian_link_by_finite_differences():
    rs = np.random.RandomState(2)
    z, y, aux = rs.randn(5, 3), rs.randn(5), np.exp(rs.randn(3))
    ll, r, c, _ = link_terms(z, y, 'gaussian', aux)
    sig = 1.0 / aux
    assert np.allclose(ll, -0.5 * ((y[:, None] - z) / sig) ** 2 - np.log(sig) - 0.5 * np.log(2 * np.pi))
    h = 1e-6
    fd = (link_terms(z + h, y, 'gaussian', aux)[0] - link_terms(z - h, y, 'gaussian', aux)[0]) / (2 * h)
    assert np.allclose(r, fd, rtol=1e-7)
    assert np.allclose(c, aux * aux)


@pytest.mark.parametrize('link', ['logistic', 'probit'])
def test_float64_links_against_mpmath(link):
    """The reference's float64 links (which the sweep tests use) to a few ulps (times the condition number for ll)
    on a grid over [-1e4, 1e4]; mpmath keeps
    log Phi(20) ~ -2.8e-89 and the probit curvature at a = -1e4 (where r (a + r) cancels to 8 digits)."""
    a = np.concatenate([-np.logspace(-3, 4, 60), [0.0], np.logspace(-3, 4, 60), [-37.5, -20.0, -6.0, -5.99, 8.0, 20.0]])
    ll, r, c, _ = link_terms(a[:, None], np.ones(a.size), link)
    assert mp_link(20.0, 'probit')[0] < -2e-89
    for i, ai in enumerate(a):
        m = mp_link(ai, link)
        tols = (ll_rtol(ai, m[0], m[1]), 1e-14, 1e-13)
        for got, want, tol in zip((ll[i, 0], r[i, 0], c[i, 0]), m, tols):
            assert abs(got - want) <= tol * abs(want) + 1e-300, (link, ai, got, want)


@pytest.mark.parametrize('N,d,S', CASES)
def test_bound_catches_the_bug_classes(N, d, S):
    """For every GPU case shape, each mutation of the reference must exceed the worst-case bound of at least one
    element, for the links the GPU test runs at that shape, with w = NULL and with AlphaDivergence-shaped weights."""
    bm = plan(d)[0]
    for link in case_links(N, S):
        X, y, theta, base, aux = make_case(N, d, S, link, case_seed(N, d, S))
        for w in (None, alpha_weights(S, S + d)):
            ref = Reference(X, y, theta, base, link, w=w, aux=aux)
            for name, dll, dgmu, dge in mutations(ref, bm):
                ratio = detected(ref, dll, dgmu, dge)
                assert ratio > 1.0, (link, name, 'weighted' if w is not None else 'w = NULL', ratio)
