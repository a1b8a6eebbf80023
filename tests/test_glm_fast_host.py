"""Host checks of the float64 reference and error model of the tensor-core GLM sweep (tests/_glm_fast_ref.py)."""
import numpy as np
import pytest

from _glm_fast_ref import (CASES, C_Z, Reference, alpha_weights, case_seed, detected, fp8_scales, make_case,
                           mutations)


def test_reference_matches_the_oracle():
    """Sign and weight conventions: ll and the weighted gradient sums against the oracle's logistic log density."""
    from oracle import viabel_oracle as vo
    N, d, S = 700, 19, 9
    X, y, theta, base = make_case(N, d, S, 5)
    w = alpha_weights(S, 3)
    ref = Reference(X, y, theta, base, w=w)
    f, g = vo.logistic_logp_grad(theta, X, y, 10.0)
    lp = -0.5 * np.sum(theta ** 2, axis=1) / 100.0 - 0.5 * d * np.log(2 * np.pi * 100.0)
    gl = g + theta / 100.0                      # likelihood part of the per-sample gradient
    assert np.allclose(ref.ll, f - lp, rtol=1e-13, atol=1e-10)
    assert np.allclose(ref.gmu, w @ gl, rtol=1e-12, atol=1e-10)
    assert np.allclose(ref.ge, np.sum(w[:, None] * gl * base, axis=0), rtol=1e-12, atol=1e-10)


def test_fp8_scales_follow_the_data():
    X, y, _, _ = make_case(1000, 64, 1, 2)
    ax, bx = fp8_scales(X, y)
    assert (ax, bx) == (2, 8)
    assert fp8_scales(X * 1024.0, y) == (ax - 10, bx + 10)


@pytest.mark.parametrize('N,d,S,general', CASES)
def test_statistical_bound_catches_the_bug_classes(N, d, S, general):
    """For every GPU case shape, each mutation of the reference must fail the statistical bound of at least one
    element (with the calibrated c_z): the thresholds detect what the tests are meant to catch."""
    X, y, theta, base = make_case(N, d, S, case_seed(N, d, S), exact=not general)
    for w in (None, alpha_weights(S, S + d)):
        ref = Reference(X, y, theta, base, w=w, exact=not general)
        for name, dll, dgmu, dge in mutations(ref):
            ratio = detected(ref, dll, dgmu, dge, c_z=C_Z)
            assert ratio > 1.0, (name, 'weighted' if w is not None else 'w = NULL', ratio)
