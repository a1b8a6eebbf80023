"""CPU: the numpy Philox reference (_philox_ref.py) that the draw-kernel tests compare against -- Random123's
known-answer vectors, the top of the 53-bit uniform, its distributions against scipy past 2^33, and the properties of
the inputs the GPU tests use that make an element-by-element comparison sound."""
import numpy as np
import pytest
from scipy import stats

import _philox_ref as pr

# Random123 kat_vectors, philox4x32_10: (key, counter c0..c3, output)
KAT = [
    (0, (0, 0, 0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    (0xffffffffffffffff, (0xffffffff,) * 4, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    (0x299f31d0a4093822, (0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
]

N_KS, START, SEED = 400000, 2 ** 33 + 1, 7
CHI2_DF = (0.3, 0.7, 1.0, 2.0, 3.0, 20.0)
T_DF = (2.5, 7.5, 40.0)


@pytest.mark.parametrize('key,ctr,out', KAT)
def test_known_answers(key, ctr, out):
    lo, hi = ctr[0] | ctr[1] << 32, ctr[2] | ctr[3] << 32
    got = pr.philox(key, np.array([lo], dtype=np.uint64), hi)
    assert tuple(int(w[0]) for w in got) == out


def test_u01_range():
    """(0, 1]: the smallest 53-bit value gives 2^-54; from 2^52 up v + 0.5 rounds to even, so the largest gives
    exactly 1.0 (as on the device)"""
    a = np.array([0, 0, 0xffffffff, 0xffffffff, 0xffffffff], dtype=np.uint64)
    b = np.array([0, 0x7ff, 0xfffff7ff, 0xfffff800, 0xffffffff], dtype=np.uint64)
    u = pr.u01_53(a, b)
    assert u[0] == u[1] == 2.0 ** -54
    assert u[2] == 1.0 - 2.0 ** -52 and u[3] == u[4] == 1.0


def test_sincospi_reduction():
    """the quadrant reduction against mpmath at the quarter points and in between"""
    import mpmath
    mpmath.mp.prec = 100
    t = np.concatenate([np.arange(9) / 4.0, np.linspace(1e-9, 2.0, 101), [2.0 ** -50, 1.0 - 2.0 ** -52]])
    sn, cs = pr._sincospi(t)

    def exact(x):                        # extended -> mpf without rounding to float64
        hi = pr.to64(x)
        return mpmath.mpf(float(hi)) + mpmath.mpf(float(pr.to64(x - hi)))

    for i, ti in enumerate(t):
        assert abs(float(mpmath.sinpi(ti) - exact(sn[i]))) <= 2.0 ** -60
        assert abs(float(mpmath.cospi(ti) - exact(cs[i]))) <= 2.0 ** -60


def test_normal_ks():
    z, _ = pr.normal_stream(SEED, START, N_KS)
    assert stats.kstest(pr.to64(z), 'norm').pvalue > 1e-3


@pytest.mark.parametrize('df', CHI2_DF)
def test_chisquare_ks_and_margins(df):
    """chi-square against scipy (df < 2 takes the shape < 1 boost, df = 2 is the a = 1 edge); df <= 3 reaches the
    v <= 0 rejection; every accept/reject decision is far from rounding"""
    x, bound, margin, vneg = pr.chisquare_stream(SEED, START, N_KS, df)
    x = pr.to64(x)
    assert np.all(x > 0) and np.all(bound < 1e-13 * np.maximum(1.0, x))
    assert stats.kstest(x, stats.chi2(df).cdf).pvalue > 1e-3
    assert margin.min() > 64
    if df <= 3:
        assert vneg > 0


@pytest.mark.parametrize('df', T_DF)
def test_student_t_ks(df):
    t, _, margin = pr.student_t_stream(SEED, START, N_KS, df)
    assert stats.kstest(pr.to64(t), stats.t(df).cdf).pvalue > 1e-3
    assert margin.min() > 64


def test_quantize():
    """bf16 and fp16 through float32, round to nearest even, against torch's conversions"""
    torch = pytest.importorskip('torch')
    rs = np.random.RandomState(3)
    x = np.concatenate([rs.randn(20000) * 10.0 ** rs.uniform(-6, 4, 20000),
                        [1 + 2.0 ** -8, 1 + 3 * 2.0 ** -9, 1 + 2.0 ** -9, 1 + 2.0 ** -24, 65520.0, -0.0]])
    xt = torch.as_tensor(x).float()
    assert np.array_equal(pr.quantize(x, 1), xt.to(torch.bfloat16).double().numpy())
    assert np.array_equal(pr.quantize(x, 2), xt.to(torch.float16).double().numpy())
