"""GPU: the Philox draw kernels (csrc/sampling.cu: vb_philox_normal_f64 / _f32, vb_philox_chisquare_f64,
vb_philox_student_t_f64) element by element against the numpy reference _philox_ref.py, at seeds with and without a
high key word, offsets up to the tail of a 1e8 x 256 stream, odd offsets, tiny counts and counts past the grid cap,
every quantisation mode and chi-square / Student-t df from the shape < 1 boost to the near-normal limit.

Every other draw consumer (the mean-field, MultivariateT and LRGaussian families, the fused step, the streaming
log-weight kernels) is tied to these kernels by its own tests, so pinning them to an independent reference pins all
of those.  A float64 value must lie within MARGIN times its derived error bound of the extended-precision reference;
a rounded output (float32, bfloat16, float16) must equal the rounded reference exactly -- an element whose reference
lies within its bound of a rounding midpoint would be ambiguous, and there are none."""
import numpy as np
import pytest
import torch

import _philox_ref as pr

pytestmark = pytest.mark.gpu

MARGIN = 1.25
SEEDS = (0, 7, 2 ** 32 + 5, 2 ** 64 - 1)
OFFSETS = (0, 1, 2 ** 32 - 1, 2 ** 33 + 1, 256 * 10 ** 8 - 7)
COUNTS = (1, 2, 3, 1001)
CHI2_DF = (0.3, 0.7, 1.0, 2.0, 3.0, 20.0, 1e4)
T_DF = (2.01, 2.5, 5.5, 40.0, 1e6)
# one thread per pair (normal) or per element, 256 threads, at most 16 blocks per SM: these counts make every
# thread take a second turn of the grid-stride loop on a B200 (148 SMs); the cases start just below a counter word
# boundary (2^32 pairs for the normal stream, 2^32 elements otherwise) so that they also cross it
WRAP_NORMAL, WRAP_GAMMA = 1300001, 700001
WRAP_SEED = 2 ** 32 + 5


@pytest.fixture(scope='module')
def vb():
    import viabel_b200
    return viabel_b200


def _cases():
    return [(s, o, n) for s in SEEDS for o in OFFSETS for n in COUNTS]


def _draw(vb, kind, n, seed, offset, df=0.0, quantize=0, f32=False):
    lib = vb._lib
    out = torch.full((n,), float('nan'), dtype=torch.float32 if f32 else torch.float64, device='cuda')
    if kind == 'normal':
        fn = lib.lib.vb_philox_normal_f32 if f32 else lib.lib.vb_philox_normal_f64
        lib.check(fn(lib.ptr(out), n, seed, offset, quantize, lib.stream()))
    elif kind == 'chi2':
        lib.check(lib.lib.vb_philox_chisquare_f64(lib.ptr(out), n, df, seed, offset, lib.stream()))
    else:
        lib.check(lib.lib.vb_philox_student_t_f64(lib.ptr(out), n, df, seed, offset, quantize, lib.stream()))
    return out.cpu().numpy().astype(np.float64)


def _check(dev, ref, bound, quantize=0, f32=False, what=''):
    """dev against the reference: within MARGIN * bound in float64, or equal to the rounded reference"""
    if quantize == 0 and not f32:
        err = pr.err64(dev, ref)
        bad = np.flatnonzero(~(err <= MARGIN * bound))
        assert bad.size == 0, '%s: %d elements off, first %d: %r vs %r (bound %.3g), worst err/bound %.3g' % (
            what, bad.size, bad[0], dev[bad[0]], pr.to64(ref[bad[0]]), bound[bad[0]], np.max(err / bound))
        return
    if quantize:
        fn = (lambda x: pr.quantize(x, quantize))
    else:
        fn = (lambda x: x.astype(np.float32).astype(np.float64))
    lo, hi = pr.rounded(ref, MARGIN * bound, fn)
    ambiguous = int(np.count_nonzero(lo != hi))
    assert ambiguous == 0, '%s: %d elements within their bound of a rounding midpoint' % (what, ambiguous)
    bad = np.flatnonzero(dev != lo)
    assert bad.size == 0, '%s: %d elements differ, first %d: %r vs %r' % (
        what, bad.size, bad[0], dev[bad[0]], lo[bad[0]])


def test_wrap_counts_pass_the_grid(vb):
    cap = 16 * 256 * vb._lib.lib.vb_device_sm_count()
    assert (WRAP_NORMAL + 1) // 2 > cap and WRAP_GAMMA > cap


@pytest.mark.parametrize('f32', [False, True], ids=['f64', 'f32'])
def test_normal_vs_reference(vb, f32):
    cases = _cases() + [(WRAP_SEED, 2 ** 33 - WRAP_NORMAL // 2, WRAP_NORMAL)]
    for seed, offset, n in cases:
        z, bound = pr.normal_stream(seed, offset, n)
        for q in (0, 1, 2):
            _check(_draw(vb, 'normal', n, seed, offset, quantize=q, f32=f32), z, bound, q, f32,
                   'seed %d offset %d n %d quantize %d' % (seed, offset, n, q))


@pytest.mark.parametrize('df', CHI2_DF)
def test_chisquare_vs_reference(vb, df):
    cases = _cases() + [(WRAP_SEED, 2 ** 32 - WRAP_GAMMA // 2, WRAP_GAMMA)]
    for seed, offset, n in cases:
        x, bound, margin, _ = pr.chisquare_stream(seed, offset, n, df)
        assert margin.min() > 64          # no accept/reject decision within reach of rounding
        _check(_draw(vb, 'chi2', n, seed, offset, df), x, bound, what='seed %d offset %d n %d' % (seed, offset, n))


@pytest.mark.parametrize('df', T_DF)
def test_student_t_vs_reference(vb, df):
    cases = _cases() + [(WRAP_SEED, 2 ** 32 - WRAP_GAMMA // 2, WRAP_GAMMA)]
    for seed, offset, n in cases:
        t, bound, margin = pr.student_t_stream(seed, offset, n, df)
        assert margin.min() > 64
        for q in (0, 1, 2):
            _check(_draw(vb, 'student', n, seed, offset, df, q), t, bound, q,
                   what='seed %d offset %d n %d quantize %d' % (seed, offset, n, q))


def test_v_nonpositive_rejection_is_compared(vb):
    """the chi-square cases at df <= 3 include draws whose first attempt is rejected at v <= 0"""
    for df in (0.3, 1.0, 3.0):
        _, _, _, vneg = pr.chisquare_stream(WRAP_SEED, 2 ** 32 - WRAP_GAMMA // 2, WRAP_GAMMA, df)
        assert vneg > 0


def test_bad_arguments(vb):
    """n < 0, a NULL output or df <= 0 -> ValueError; n = 0 is a no-op"""
    lib = vb._lib
    out = torch.empty(4, dtype=torch.float64, device='cuda')
    calls = {
        'normal': lambda p, n, df: lib.lib.vb_philox_normal_f64(p, n, 1, 0, 0, lib.stream()),
        'normal32': lambda p, n, df: lib.lib.vb_philox_normal_f32(p, n, 1, 0, 0, lib.stream()),
        'chi2': lambda p, n, df: lib.lib.vb_philox_chisquare_f64(p, n, df, 1, 0, lib.stream()),
        'student': lambda p, n, df: lib.lib.vb_philox_student_t_f64(p, n, df, 1, 0, 0, lib.stream()),
    }
    for name, call in calls.items():
        bad = [(lib.ptr(out), -1, 3.0), (None, 4, 3.0)]
        if name in ('chi2', 'student'):
            bad += [(lib.ptr(out), 4, 0.0), (lib.ptr(out), 4, float('nan'))]
        for p, n, df in bad:
            with pytest.raises(ValueError):
                lib.check(call(p, n, df))
        lib.check(call(None, 0, 3.0))
