"""Host mirror of the PSIS threshold pipeline in viabel_b200/csrc/psis.cu, the named edge cases built to reach each of
its branches, and a wrapper of the oracle (numpy only, shared by the CPU and GPU tests).

The mirror follows psis_plan, psis_sample_select_kernel and the candidate histogram of pass A / gather kernel with the
same double arithmetic, key order and casts, so that it predicts which path a sampled (exact=False) run takes: the
candidate threshold t0, the candidate count C (the device's result slot R_NCAND), status 1, the boundary bin and its
population.  Each case carries the branch labels of BRANCHES it is built for.
"""
import math

import numpy as np

from _problems import _t_ratio, psis_case

kSampleMax, kSelThreads, kBins, kGather = 16384, 1024, 2048, 8192

BRANCHES = ('t0=-inf', 'sample16', 'sample1_max', 'sample1_exact', 'members<=1024', 'members<=8192',
            'members>8192', 'scale0', 'status1_overflow', 'status1_few')

_TOP = np.uint64(1 << 63)


def dkey(x):
    """Order-preserving 64-bit key of a double (psis.cu dkey): -0.0 sorts below +0.0."""
    b = np.ascontiguousarray(x, dtype=np.float64).view(np.uint64)
    return np.where(b >> np.uint64(63), ~b, b | _TOP)


def dkey_inv(k):
    k = np.uint64(k)
    b = (k & ~_TOP) if (k >> np.uint64(63)) else ~k
    return float(np.array([b], dtype=np.uint64).view(np.float64)[0])


def plan(n, reff=1.0, n_global=None, world=1):
    """psis_plan: tail length M, sample size and stride, sample rank R, candidate capacity."""
    n_global = n if n_global is None else n_global
    M = int(math.ceil(min(0.2 * float(n_global), 3.0 * math.sqrt(float(n_global) / reff))))
    m = min(n, kSampleMax)
    stride = n // m
    f = float(M + 1) * float(m) / float(n)
    R = float(math.ceil(f + 8.0 * math.sqrt(f) + 16.0))
    if m == n:
        R = float(M + 1)
    R = min(R, float(n))
    R = int(min(R, 4.0e9))
    cap = 4.0 * (float(R) * float(n) / float(m)) + 65536.0
    cap = min(cap, float(n))
    if cap < float(M + 1) <= float(n):
        cap = float(M + 1)
    cap = int(min(max(cap, float(world) * (M + 1) if world > 1 else 0.0), 4.0e9))
    return dict(M=M, m=m, stride=stride, R=R, cap=cap)


def sample_positions(n):
    p = plan(n)
    return np.arange(p['m'], dtype=np.int64) * p['stride']


def _kth_largest(keys, K):
    return np.sort(keys)[::-1][K - 1]


def sample_select(sample, R):
    """psis_sample_select_kernel on the m strided sample values: (t0, sample maximum, path label)."""
    m = sample.size
    if R >= m:
        return -math.inf, -math.inf, 't0=-inf'
    keys = dkey(sample)
    if R <= 256 and m == kSampleMax:
        # 16 CTAs: maxima of 16 consecutive entries, 3 radix digits (stop_shift 31): lower bound of the bucket
        gm = keys.reshape(kSampleMax // 16, 16).max(axis=1)
        k = _kth_largest(gm, R) & ~np.uint64((1 << 31) - 1)
        return dkey_inv(k), dkey_inv(gm.max()), 'sample16'
    # one CTA: thread t holds the keys of entries u * 1024 + t (key 0, i.e. no entry, is below everything)
    pad = np.zeros(kSampleMax, dtype=np.uint64)
    pad[:m] = keys
    kmax = pad.reshape(16, kSelThreads).max(axis=0)
    hi = dkey_inv(kmax.max())
    if R <= 256:
        return dkey_inv(_kth_largest(kmax[kmax != 0], R)), hi, 'sample1_max'
    return dkey_inv(_kth_largest(keys[keys != 0], R)), hi, 'sample1_exact'


def cbin(x, lo, scale):
    """Linear candidate bins over [t0, sample maximum]: (x - lo) * scale truncated toward zero, clamped."""
    with np.errstate(all='ignore'):
        f = (np.asarray(x, dtype=np.float64) - lo) * scale
        b = np.where(f >= kBins, kBins - 1, np.where(f > 0, np.trunc(f), 0.0))      # NaN -> 0, as cvt.rzi.s32
    return b.astype(np.int64)


def mirror_parts(n, sample, candidates_ge, reff=1.0, n_global=None, world=1):
    """The sampled run of a device call on n draws whose m strided sample values are `sample`;
    candidates_ge(t0) returns the draws x >= t0 (every draw when t0 = -inf)."""
    p = plan(n, reff, n_global, world)
    M, R, cap = p['M'], p['R'], p['cap']
    t0, hi, path = sample_select(np.asarray(sample, dtype=np.float64), R)
    cand = np.asarray(candidates_ge(t0), dtype=np.float64)
    C = int(cand.size)
    res = dict(p, t0=t0, hi=hi, path=path, C=C, status=0, bstar=None, need=None, members=None, scale=None)
    labels = {path}
    if C > cap:
        res['status'] = 1
        labels.add('status1_overflow')
    elif C < M + 1:
        res['status'] = 1
        labels.add('status1_few')
    else:
        with np.errstate(over='ignore'):
            scale = float(kBins) / (hi - t0) if (t0 > -math.inf and hi > t0) else 0.0
        b = cbin(cand, t0, scale) if scale > 0.0 else np.zeros(C, dtype=np.int64)
        h = np.bincount(b, minlength=kBins)
        cum = np.cumsum(h[::-1])
        j = int(np.searchsorted(cum, M + 1))              # first bin from the top whose cumulative count reaches M+1
        bstar = kBins - 1 - j
        members = int(h[bstar])
        res.update(scale=scale, bstar=bstar, need=int(M + 1 - (cum[j] - members)), members=members)
        if scale == 0.0:
            labels.add('scale0')
        labels.add('members<=1024' if members <= kSelThreads else
                   'members<=8192' if members <= kGather else 'members>8192')
    res['labels'] = frozenset(labels)
    return res


def mirror(lw, reff=1.0, n_global=None, world=1):
    """Prediction for the sampled run of vb_psislw_f64 (or one shard's vb_psis_dist_local) on the array lw."""
    lw = np.asarray(lw, dtype=np.float64)
    n = lw.size
    p = plan(n, reff, n_global, world)
    sample = lw[np.arange(p['m'], dtype=np.int64) * p['stride']]
    return mirror_parts(n, sample, lambda t0: lw if t0 == -math.inf else lw[lw >= t0], reff, n_global, world)


# ---- oracle -----------------------------------------------------------------------------------------------------
def oracle(lw, reff=1.0):
    """oracle.viabel_oracle.psislw_1d with the quantities the device reports: out, k, xcut (shifted cutoff), lse,
    max, n2, the tail indices in (value, index) order, and the moments sum v, sum exp(2 v) of v = out + lse."""
    from oracle import viabel_oracle as vo
    lw = np.asarray(lw, dtype=np.float64)
    with np.errstate(all='ignore'):
        out, k, tail, _ = vo.psislw_1d(lw, reff, return_tail=True)
        mx = np.max(lw)
        x = lw - mx
        M = vo.psis_tail_len(lw.size, reff)
        kth = lw.size - M - 1
        xcut = max(np.partition(x, kth)[kth], math.log(np.finfo(float).tiny))
        tail_ord = tail[np.lexsort((tail, x[tail]))]          # (value, index) order, also when n2 <= 4
        # the log-sum-exp psislw_1d subtracts: its smoothed, unnormalised weights rebuilt with the same calls
        if k >= 1.0 / 3.0 and not np.isinf(k):
            expcut = math.exp(xcut)
            k2, sigma = vo.gpdfit(np.exp(x[tail_ord]) - expcut)
            assert k2 == k
            x[tail_ord] = np.log(vo.gpinv((np.arange(tail_ord.size) + 0.5) / tail_ord.size, k, sigma) + expcut)
            x[x > 0] = 0.0
        lse = float(vo.sumlogs(x))
        v = out + lse
        sumv, sume2 = float(v.sum()), float(np.exp(2.0 * v).sum())
    return dict(out=out, k=float(k), xcut=float(xcut), lse=lse, max=float(mx), n2=int(tail_ord.size),
                tail=np.asarray(tail_ord, dtype=np.int64), sumv=sumv, sumexp2v=sume2, M=M)


# ---- Reff at which the tail length is a given M ------------------------------------------------------------------
def reff_for_tail(n, M):
    """A Reff with psis_tail_len(n, Reff) == M (M < 0.2 n): 3 sqrt(n / Reff) = M - 1/2."""
    from oracle import viabel_oracle as vo
    reff = 9.0 * n / (M - 0.5) ** 2
    assert vo.psis_tail_len(n, reff) == M, (n, M, reff)
    return reff


REFF_TAILS = (4, 5, 6, 255, 256, 257, 1023, 1024, 1025, 2047, 2048, 2049, 4096, 4097)
REFF_VALUES = (0.01, 0.3, 7.5, 1e6)


def reff_cases():
    """(name, Reff) on big_1e6: tail lengths at the kernels' fixed sizes, and a few plain values of Reff."""
    cases = [('n2_%d' % M, reff_for_tail(1000000, M)) for M in REFF_TAILS]
    return cases + [('reff_%g' % r, r) for r in REFF_VALUES]


# ---- named cases --------------------------------------------------------------------------------------------------
def _rank_desc(x):
    return np.argsort(-x, kind='stable')


def _outlier(delta, pos):
    x = psis_case('big_1e6').copy()
    x[pos] = x.max() + delta
    return x


def _sorted(n, descending):
    x = np.sort(_t_ratio(n, 4, 9, 100 + n % 997))
    return x[::-1].copy() if descending else x


def _outlier_1e7():
    rs = np.random.RandomState(21)
    x = rs.standard_normal(10000000)
    x[0] = x.max() + 1e4                    # a sampled index: the candidate bins become 5 units wide
    return x


def _tie_block(width):
    x = psis_case('big_1e6').copy()
    M = plan(x.size)['M']
    r = _rank_desc(x)
    lo = M - min(width // 2, M // 2)
    x[r[lo:lo + width]] = x[r[M]]
    return x


def _periodic(high):
    n = 2000000
    rs = np.random.RandomState(22 + high)
    x = rs.standard_t(4, n)
    s = sample_positions(n)
    x[s] = (60.0 if high else -60.0) + rs.rand(s.size)
    return x


def _signed_zeros():
    x = _t_ratio(100000, 5, 7, 23)
    M = plan(x.size)['M']
    x -= np.sort(x)[::-1][M]                # the value at rank M+1 becomes 0
    r = _rank_desc(x)
    blk = r[M - 40:M + 40]
    x[blk] = np.where(np.arange(blk.size) % 2 == 0, 0.0, -0.0)
    return x


def _huge_pm():
    """-1e308 at the sampled positions, +1e308 at one of them, a few finite sampled draws, -1.5e308 elsewhere: the
    sample threshold is -1e308, hi - t0 overflows (no linear bins) and x - max is -inf for every finite x."""
    n = 100000
    rs = np.random.RandomState(24)
    x = np.full(n, -1.5e308)
    s = sample_positions(n)
    x[s] = -1e308
    x[s[rs.choice(s.size, 200, replace=False)]] = rs.standard_t(3, 200)
    x[s[7]] = 1e308
    return x


def _huge_one():
    x = _t_ratio(100000, 5, 7, 25)
    x[0] = 1e308
    return x


def _pos_inf():
    x = _t_ratio(100000, 5, 7, 26)
    x[[0, 777]] = np.inf                    # one sampled, one not: the sample maximum is +inf
    return x


def _ulp_above():
    """Tail draws set one ulp above the (M+1)-th largest c.  Shifted by the maximum they equal c - max, so they are
    not in the tail {x - max > c - max}."""
    x = _t_ratio(100000, 5, 7, 27)
    M = plan(x.size)['M']
    r = _rank_desc(x)
    x = x - x[r[M]] + 0.3                   # c = 0.3 with a maximum of a few units: the shift rounds away the ulp
    c = x[r[M]]
    up = np.nextafter(c, np.inf)
    x[r[M - 200:M]] = up
    mx = x.max()
    assert up - mx == c - mx and up > c
    return x


def _sorted_shard_mix():
    a = _t_ratio(1000000, 4, 9, 28)
    return np.concatenate([a, np.sort(_t_ratio(1000000, 4, 9, 29))])


NAMED = {
    'sorted_asc_20000': (lambda: _sorted(20000, False), {'sample1_exact', 'members<=8192'}),
    'sorted_desc_20000': (lambda: _sorted(20000, True), {'sample1_exact', 'members<=1024'}),
    'sorted_asc_30000': (lambda: _sorted(30000, False), {'sample1_exact', 'members>8192'}),
    'sorted_desc_30000': (lambda: _sorted(30000, True), {'sample1_exact', 'status1_few'}),
    'sorted_asc_1e5': (lambda: _sorted(100000, False), {'sample1_exact', 'members<=8192'}),
    'sorted_desc_1e5': (lambda: _sorted(100000, True), {'sample1_exact', 'members<=1024'}),
    'sorted_asc_1e6': (lambda: _sorted(1000000, False), {'sample16', 'status1_overflow'}),
    'sorted_desc_1e6': (lambda: _sorted(1000000, True), {'sample16', 'status1_overflow'}),
    'outlier_40_sampled': (lambda: _outlier(40.0, 0), {'sample16', 'members<=1024'}),
    'outlier_200_sampled': (lambda: _outlier(200.0, 0), {'sample16', 'members<=1024'}),
    'outlier_1e4_sampled': (lambda: _outlier(1e4, 0), {'sample16', 'members<=8192'}),
    'outlier_1e4_unsampled': (lambda: _outlier(1e4, 5), {'sample16', 'members<=1024'}),
    'outlier_1e7': (_outlier_1e7, {'sample16', 'members>8192'}),
    'tie_block_4000': (lambda: _tie_block(4000), {'sample16', 'members<=8192'}),
    'tie_block_20000': (lambda: _tie_block(20000), {'sample16', 'members>8192'}),
    'periodic_low': (lambda: _periodic(False), {'sample16', 'status1_overflow'}),
    'periodic_high': (lambda: _periodic(True), {'sample16', 'status1_few'}),
    'signed_zeros': (_signed_zeros, {'sample1_exact', 'members<=1024'}),
    'huge_pm_1e308': (_huge_pm, {'sample1_exact', 'scale0', 'members>8192'}),
    'huge_1e308': (_huge_one, {'sample1_exact', 'members<=8192'}),
    'pos_inf': (_pos_inf, {'sample1_exact', 'scale0', 'members<=8192'}),
    'ulp_above_cutoff': (_ulp_above, {'sample1_exact', 'members<=1024'}),
    'sorted_shard_mix': (_sorted_shard_mix, {'sample16', 'members<=1024'}),
}

SMALL_KINDS = ('distinct', 'three_values', 'all_equal')
SMALL_N = tuple(range(2, 65))


def small_case(kind, n):
    rs = np.random.RandomState(1000 + n)
    if kind == 'distinct':
        return rs.standard_t(3, n)
    if kind == 'three_values':
        return np.array([-1.5, 0.25, 2.0])[rs.randint(0, 3, n)]
    return np.full(n, 0.75)


_cache = {}


def named_case(name):
    if name not in _cache:
        _cache[name] = NAMED[name][0]()
    return _cache[name]


# ---- more than 2^31 draws ----------------------------------------------------------------------------------------
BIG_N = 2 ** 31 + 2 ** 20 + 3
BIG_PIECE = 8000000            # enough piece draws in the 1-in-131 136 sample for the 26th of 1024 group maxima
BIG_GAP = 900.0                # the body sits this far below the piece: its exponentials underflow


def big_piece():
    """(positions, values, body value) of the 2^31-draw case: t-ratio draws at seeded distinct positions, the
    largest of them moved past index 2^31; every other draw is the body value."""
    if 'big' not in _cache:
        rs = np.random.RandomState(30)
        pos = np.unique(rs.randint(0, BIG_N, size=BIG_PIECE, dtype=np.int64))
        vals = _t_ratio(pos.size, 4, 9, 31)
        late = np.flatnonzero(pos >= 2 ** 31)
        top = np.argsort(vals)[::-1][:late.size // 2]
        top = top[pos[top] < 2 ** 31]
        late = late[~np.isin(late, top)][:top.size]
        vals[top], vals[late] = vals[late].copy(), vals[top].copy()
        _cache['big'] = (pos, vals, float(vals.min() - BIG_GAP))
    return _cache['big']


def mirror_big():
    pos, vals, body = big_piece()
    p = plan(BIG_N)
    sample = np.full(p['m'], body)
    hit = (pos % p['stride'] == 0) & (pos // p['stride'] < p['m'])
    sample[pos[hit] // p['stride']] = vals[hit]

    def cand(t0):
        assert body < t0
        return vals[vals >= t0]
    return mirror_parts(BIG_N, sample, cand)


def big_surrogate(n_body=16):
    """The piece followed by a few body draws, with Reff' = n' / n: the same tail length M, maximum, cutoff and tail
    (surrogate index j < piece size is draw pos[j]) as the full array."""
    pos, vals, body = big_piece()
    sur = np.concatenate([vals, np.full(n_body, body)])
    return sur, sur.size / BIG_N, pos
