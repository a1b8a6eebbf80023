"""numpy reference of the Philox4x32-10 draw streams (csrc/common.cuh, csrc/philox_draws.cuh, csrc/sampling.cu),
independent of the library.

The integer part (Philox, the 53-bit uniforms, stream ids, counters, attempt numbering) is bit-exact with the device
code.  Everything after the uniforms is evaluated in extended precision (np.longdouble when it carries at least a
64-bit mantissa, else mpmath at 80 bits), and each value comes with a first-order bound on the error of the device's
float64 evaluation, derived from CUDA's documented ulp bounds: log 1 ulp, log1p 1 ulp, exp 1 ulp, sincospi 2 ulp,
pow 2 ulp, and correctly rounded + - * / sqrt.  A device value that differs from the reference by more than its bound
(times a small margin) is a wrong value, not rounding.

Stream layout (element e of a stream is a pure function of (seed, e)):
  normal      element e: component e & 1 of the Box-Muller pair at counter e >> 1, stream id 0
  chi-square  element e: 2 gamma(df / 2) at counter e, stream id 1
  Student-t   element e: z0 of the pair at (e, stream id 2) / sqrt(2 gamma(df / 2) at (e, stream id 3) / df)
  gamma attempt k at (e, sid): normal from sid | (2k + 1) << 40, uniform from sid | (2k + 2) << 40; shape < 1 adds
  the boost u^(1/a) with u from sid | 1 << 62 (Marsaglia-Tsang)."""
import numpy as np

U = 2.0 ** -53                       # float64 unit roundoff; 1 ulp <= 2 U |x|
_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
_MASK = np.uint64(0xFFFFFFFF)
_S32 = np.uint64(32)

# ---- extended precision ------------------------------------------------------------------------------------------
EXTENDED = np.finfo(np.longdouble).nmant >= 63
if EXTENDED:
    XF = np.longdouble
    _PI = 4 * np.arctan(np.longdouble(1))

    def xf(x):
        return np.asarray(x, dtype=np.longdouble)

    _log, _log1p, _sqrt, _sin, _cos, _exp, _pow = np.log, np.log1p, np.sqrt, np.sin, np.cos, np.exp, np.power
else:                                # pragma: no cover - platforms whose long double is float64
    import mpmath
    mpmath.mp.prec = 80
    XF = object
    _PI = mpmath.pi

    def xf(x):
        return np.frompyfunc(mpmath.mpf, 1, 1)(np.asarray(x, dtype=np.float64)).astype(object)

    _log, _log1p, _sqrt, _sin, _cos, _exp = (np.frompyfunc(f, 1, 1) for f in (
        mpmath.log, mpmath.log1p, mpmath.sqrt, mpmath.sin, mpmath.cos, mpmath.exp))
    _pow = np.frompyfunc(mpmath.power, 2, 1)


def to64(x):
    """extended -> nearest float64"""
    return np.asarray(x).astype(np.float64)


def abs64(x):
    return np.abs(to64(x)) if XF is object else np.abs(np.asarray(x)).astype(np.float64)


def err64(dev, ref):
    """|dev - ref| in float64, the difference taken in extended precision"""
    return abs64(xf(dev) - ref)


# ---- Philox4x32-10 and the 53-bit uniform -------------------------------------------------------------------------
def philox(seed, ctr_lo, ctr_hi):
    """Philox4x32-10 of counter (ctr_lo, ctr_hi) = words (c0, c1, c2, c3) under key (seed low, seed high), vectorised
    over uint64 arrays; four uint64 arrays of 32-bit words (common.cuh Philox::operator())."""
    lo = np.asarray(ctr_lo, dtype=np.uint64)
    hi = np.broadcast_to(np.asarray(ctr_hi, dtype=np.uint64), lo.shape)
    c0, c1, c2, c3 = lo & _MASK, lo >> _S32, hi & _MASK, hi >> _S32
    seed = int(seed)
    k0, k1 = np.uint64(seed & 0xFFFFFFFF), np.uint64(seed >> 32)
    for _ in range(10):
        p0, p1 = _M0 * c0, _M1 * c2          # < 2^64: exact in uint64
        c0, c1, c2, c3 = (p1 >> _S32) ^ c1 ^ k0, p1 & _MASK, (p0 >> _S32) ^ c3 ^ k1, p0 & _MASK
        k0, k1 = (k0 + _W0) & _MASK, (k1 + _W1) & _MASK
    return c0, c1, c2, c3


def u01_53(a, b):
    """the device's (((a << 32) | b) >> 11) + 0.5) * 2^-53 in float64, in (0, 1]: for the top 53-bit values the + 0.5
    rounds to even, so (0xffffffff, 0xffffffff) gives exactly 1.0"""
    v = ((np.asarray(a, dtype=np.uint64) << _S32) | np.asarray(b, dtype=np.uint64)) >> np.uint64(11)
    return (v.astype(np.float64) + 0.5) * (1.0 / 9007199254740992.0)


# ---- Box-Muller --------------------------------------------------------------------------------------------------
def _sincospi(t):
    """(sin(pi t), cos(pi t)) in extended precision for float64 t in [0, 2]: t = k / 2 + r exactly, |r| <= 1/4"""
    k = np.rint(2.0 * t)
    r = t - 0.5 * k                      # exact (Sterbenz)
    s, c = _sin(_PI * xf(r)), _cos(_PI * xf(r))
    q = k.astype(np.int64) & 3
    sn = np.where(q == 0, s, np.where(q == 1, c, np.where(q == 2, -s, -c)))
    cs = np.where(q == 0, c, np.where(q == 1, -s, np.where(q == 2, -c, s)))
    return sn, cs


EPS_NORMAL = 7 * U                   # log 1 ulp (halved by sqrt) + sqrt + sincospi 2 ulp + the product


def normal_pair(seed, ctr, sid):
    """Box-Muller pair (z0, z1) at (counter ctr, stream id sid): extended-precision values; each has relative error
    bound EPS_NORMAL in float64 on the device (the uniforms are exact)"""
    r = philox(seed, ctr, sid)
    u1, u2 = u01_53(r[0], r[1]), u01_53(r[2], r[3])
    rad = _sqrt(-2 * _log(xf(u1)))
    sn, cs = _sincospi(2.0 * u2)
    return rad * cs, rad * sn


def normal_stream(seed, offset, n):
    """elements offset .. offset + n - 1 of the standard-normal stream: (values, float64 error bound)"""
    e = np.uint64(offset) + np.arange(n, dtype=np.uint64)
    z0, z1 = normal_pair(seed, e >> np.uint64(1), 0)
    z = np.where((e & np.uint64(1)) == 1, z1, z0)
    return z, EPS_NORMAL * abs64(z)


# ---- Marsaglia-Tsang gamma ---------------------------------------------------------------------------------------
def gamma(seed, elem, sid, a):
    """gamma(shape a) at counters elem of stream id sid.  Returns (values, relative error bound, acceptance margin,
    number of v <= 0 rejections).  dd, c and 1/a are the device's float64 expressions, so they are the same numbers
    here.  The margin of a draw is the smallest |log u - rhs| over its attempts in units of that decision's rounding
    reach U (x^2 + dd (1 + v^3 + |log v^3|) + |log u|): rhs sums terms of size dd that cancel, so at large shape the
    device's rhs is off by O(dd U), not O(U).  A margin far above 1 means the device decides every attempt as the
    reference does."""
    elem = np.asarray(elem, dtype=np.uint64)
    n = elem.shape[0]
    a = float(a)
    boost, eps_boost = xf(np.ones(n)), 0.0
    if a < 1.0:
        r = philox(seed, elem, sid | (1 << 62))
        boost = _pow(xf(u01_53(r[0], r[1])), xf(1.0 / a))
        eps_boost = 4 * U                # pow 2 ulp
        a += 1.0
    dd = a - 1.0 / 3.0
    c = 1.0 / np.sqrt(9.0 * dd)
    val = xf(np.zeros(n))
    eps = np.full(n, np.inf)
    margin = np.full(n, np.inf)
    vneg = 0
    todo = np.arange(n)
    for attempt in range(64):
        if todo.size == 0:
            break
        x, _ = normal_pair(seed, elem[todo], sid | ((2 * attempt + 1) << 40))
        v = 1 + c * x
        ok = to64(v) > 0
        vneg += int((~ok).sum())
        idx, x, v = todo[ok], x[ok], v[ok]
        v3 = v * v * v
        r = philox(seed, elem[idx], sid | ((2 * attempt + 2) << 40))
        lu, lv = _log(xf(u01_53(r[0], r[1]))), _log(v3)
        rhs = 0.5 * x * x + dd - dd * v3 + dd * lv
        reach = U * (abs64(x * x) + dd * (1 + abs64(v3) + abs64(lv)) + abs64(lu))
        margin[idx] = np.minimum(margin[idx], abs64(lu - rhs) / reach)
        acc = to64(lu - rhs) < 0
        ia = idx[acc]
        val[ia] = boost[ia] * dd * v3[acc]
        # v = fl(1 + c x) (fused or not): c |x| (EPS_NORMAL + U) + U |v|; v^3 triples it plus two products; then the
        # product with boost * dd
        eps_v = (c * abs64(x[acc]) * (EPS_NORMAL + U) + U * abs64(v[acc])) / abs64(v[acc])
        eps[ia] = eps_boost + 3 * eps_v + 4 * U
        todo = np.setdiff1d(todo, ia, assume_unique=True)
    assert todo.size == 0, 'no acceptance in 64 attempts'
    return val, eps, margin, vneg


def chisquare_stream(seed, offset, n, df):
    """elements offset .. offset + n - 1 of the chi-square stream: (values, error bound, margin, v <= 0 count)"""
    e = np.uint64(offset) + np.arange(n, dtype=np.uint64)
    g, eps, margin, vneg = gamma(seed, e, 1, 0.5 * df)
    x = 2 * g
    return x, eps * abs64(x), margin, vneg


def student_t_stream(seed, offset, n, df):
    """elements offset .. offset + n - 1 of the Student-t stream: (values, error bound, margin)"""
    e = np.uint64(offset) + np.arange(n, dtype=np.uint64)
    z, _ = normal_pair(seed, e, 2)
    g, eps_g, margin, _ = gamma(seed, e, 3, 0.5 * df)
    t = z / _sqrt(2 * g / df)
    eps = EPS_NORMAL + 0.5 * (eps_g + U) + 2 * U               # chi2 / df, sqrt, the quotient
    return t, eps * abs64(t), margin


# ---- quantisation ------------------------------------------------------------------------------------------------
def bf16_rn(x32):
    """float32 -> bfloat16 (round to nearest even, by bits) as float32"""
    b = np.asarray(x32, dtype=np.float32).view(np.uint32)
    b = (b + np.uint32(0x7FFF) + ((b >> np.uint32(16)) & np.uint32(1))) & np.uint32(0xFFFF0000)
    return b.view(np.float32)


def quantize(x, mode):
    """the device's quantize_draw on float64 x: 1 = bfloat16, 2 = float16, both through float32 first"""
    x32 = np.asarray(x, dtype=np.float64).astype(np.float32)
    with np.errstate(over='ignore'):
        return (x32.astype(np.float16) if mode == 2 else bf16_rn(x32)).astype(np.float64)


def rounded(ref, bound, fn):
    """fn (a monotone rounding of float64) at both ends of [ref - bound, ref + bound]: (low, high).  Where they agree
    the device must give exactly that value; where they differ the reference lies within its error bound of a
    rounding midpoint (an ambiguous element) and either neighbour is right."""
    r = to64(ref)
    with np.errstate(over='ignore'):
        return fn(np.nextafter(r - bound, -np.inf)), fn(np.nextafter(r + bound, np.inf))
