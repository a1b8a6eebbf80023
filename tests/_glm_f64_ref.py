"""Float64 reference of the exact GLM kernels (vb_glm_sweep_f64, vb_glm_link_f64, vb_glm_point_f64) and the
worst-case error model of the sweep; mpmath values of the links at one point.

With z_ns = x_n.theta_s, a_ns = y_n z_ns (logistic / probit), r_ns = dloglik/dz and c_ns = -d^2 loglik/dz^2 the
sweep returns
    ll[s]  = sum_n loglik(y_n, z_ns)
    gmu[j] = sum_n x_nj sum_s w_s r_ns
    ge[j]  = sum_n x_nj sum_s w_s r_ns e_sj
The reference computes z with float64 GEMMs over row chunks and the links with formulas that do not cancel
(sigmoid of both signs, scipy's log_ndtr and erfcx, the continued fraction of the Mills ratio below a = -6).

Worst-case bound per element, from the kernel's numerics (glm_f64.cu):
  z     |dz_ns| <= c_z u A_ns,  A_ns = sum_j |x_nj theta_sj|     (device DMMA and the reference GEMM together)
  link  |dll_ns| <= |r_ns| dz_ns + c_l u M_ns,  M_ns = the sum of the magnitudes of the terms of loglik;
        |dr_ns| <= c_ns dz_ns + c_l u |r_ns|
  sums  u n_sum per addition chain: the device adds ll over MT rows of each of ceil(tiles / grid) tiles, three shuffle
        levels and 148 CTA partials (N / 1184 + 160 terms at most), gmu / ge over BM rows, the tiles and the partials,
        r w over S samples
  back-projections: |x_nj| and |e_sj| weight the perturbations of r.
c_z and c_l are calibrated on a B200 (DESIGN.md 2 lists the largest err / bound measured per output).
"""
import numpy as np
from scipy import special

C_Z = 16.0
C_L = 8.0
U = 2.0 ** -53
LOG2PI = float(np.log(2.0 * np.pi))
LINKS = ('logistic', 'probit', 'gaussian')
LINK_ID = {'logistic': 0, 'probit': 1, 'gaussian': 2}
SMEM = 227 * 1024


# ---- the sweep's plan (make_plan in glm_f64.cu) ---------------------------------------------------------------------
def plan(d):
    """(BM, priv) of the sweep at dimension d, or None where it returns VB_ERR_UNSUPPORTED."""
    KG = -(-d // 8)
    Dp = KG * 8
    P = Dp + 8 if Dp % 16 == 0 else Dp + 16
    warps = 16
    for bm in (32, 16, 8):
        smem = 8 * (bm * P + 2 * bm + 2 * Dp)
        if smem <= SMEM:
            priv = smem + 8 * ((warps - 1) * Dp + warps * bm) <= SMEM
            if not priv and warps * bm > Dp and smem + 8 * (warps * bm - Dp) > SMEM:
                return None
            return bm, priv
    return None


# ---- links in float64 ------------------------------------------------------------------------------------------------
def mills_tail(x):
    """a + r at a = -x, x > 6 (r = phi(a) / Phi(a)): 1 / (x + 2 / (x + 3 / (x + ...))), 24 terms."""
    t = np.zeros_like(x)
    for k in range(24, 1, -1):
        t = k / (x + t)
    return 1.0 / (x + t)


def link_terms(z, y, link, aux=None):
    """Per element: ll, r = dll/dz, c = -d^2 ll / dz^2 and M (magnitude of ll's terms).  z [n, S], y [n], aux [S]."""
    z = np.asarray(z, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)[:, None]
    if link == 'gaussian':
        e = (y - z) * aux
        ll = -0.5 * e * e + np.log(aux) - 0.5 * LOG2PI
        return ll, e * aux, np.broadcast_to(aux * aux, z.shape), 0.5 * e * e + np.abs(np.log(aux)) + 1.0
    a = y * z
    if link == 'logistic':
        ll = -np.logaddexp(0.0, -a)
        dl = special.expit(-a)
        c = special.expit(a) * dl
        return ll, y * dl, c, np.abs(ll)
    ll = np.where(a > 0, np.log1p(-special.ndtr(-np.abs(a))), special.log_ndtr(a))
    with np.errstate(over='ignore', under='ignore', divide='ignore', invalid='ignore'):
        dl = np.where(a < 0, np.sqrt(2.0 / np.pi) / special.erfcx(-a / np.sqrt(2.0)),
                      (np.exp(-0.5 * np.asarray(a, dtype=np.longdouble) ** 2) / np.sqrt(2.0 * np.pi)).astype(np.float64)
                      / special.ndtr(a))
        x = np.maximum(-a, 6.0)
        c = np.where(a >= -6.0, dl * (a + dl), dl * mills_tail(x))
    return ll, y * dl, c, np.abs(ll) + 1.0


# ---- mpmath at one point ---------------------------------------------------------------------------------------------
def mp_link(a, link):
    """(ll, dl, c) of the logistic / probit link at a = y z to about 30 digits, as floats."""
    import mpmath as mp
    # digits lost to the cancellation of a + r grow like 2 log10 |a|; mpmath's exponent range keeps Phi(-20) ~ 2.8e-89
    with mp.workdps(40 + 2 * int(np.log10(1.0 + abs(float(a))))):
        a = mp.mpf(float(a))
        if link == 'logistic':
            ea = mp.exp(a)
            ll = -mp.log1p(1 / ea)
            dl = 1 / (1 + ea)
            c = ea / (1 + ea) ** 2
        else:
            P = mp.ncdf(a)
            ll = mp.log1p(-mp.ncdf(-a)) if a > 0 else mp.log(P)
            dl = mp.npdf(a) / P
            c = dl * (a + dl)
        return float(ll), float(dl), float(c)


def ll_rtol(a, ll, dl, ulps=1e-14):
    """Relative tolerance of a float64 log-likelihood at a: `ulps` times its condition number 1 + |a dl / ll|
    (log Phi(a) in the right tail, ~ -phi(a) / a, turns the rounding of a / sqrt 2 in erfc into an error ~ u a^2)."""
    with np.errstate(divide='ignore', invalid='ignore'):
        k = np.where(ll != 0, np.abs(np.asarray(a) * dl / np.where(ll != 0, ll, 1.0)), 0.0)
    return ulps * (1.0 + k)


# ---- seeded cases ----------------------------------------------------------------------------------------------------
def make_case(N, d, S, link, seed, saturate=True):
    """X, y, theta, base, aux of one sweep: logits of order one, plus up to four rows (none of the last
    tile's, nor row N // 2) scaled so that |a| reaches 40, 300 and 1e3 (saturated links)."""
    rs = np.random.RandomState(seed)
    X = rs.randn(N, d)
    beta = rs.randn(d) / np.sqrt(d)
    base = rs.randn(S, d)
    theta = beta + base / (2.0 * np.sqrt(d))
    z = X @ beta
    if link == 'gaussian':
        y = z + rs.randn(N)
    else:
        p = special.ndtr(z) if link == 'probit' else special.expit(z)
        y = np.where(rs.rand(N) < p, 1.0, -1.0)
    if saturate and N >= 8:
        for n, target in zip((1, 2, 3, N // 3), (1e3, 300.0, 40.0, 1e3)):
            m = np.max(np.abs(theta @ X[n]))
            if m > 0:
                X[n] *= target / m
    aux = np.exp(0.3 * rs.randn(S))
    return X, y, theta, base, aux


def alpha_weights(S, seed):
    """AlphaDivergence-shaped weights (max exactly 1) with exact zeros and values down to 1e-30."""
    rs = np.random.RandomState(seed)
    w = np.exp(-rs.exponential(2.0, S))
    w[rs.randint(S)] = 1.0
    if S > 2:
        w[1::7] = 0.0
        w[2::11] = 1e-30
        w[int(np.argmax(w))] = 1.0
    return w


def n_sum(N):
    return N / 1184.0 + 200.0


class Reference(object):
    """ll / gmu / ge of the sweep in float64 and their worst-case bounds (c_z, c_l applied in `bounds`)."""

    def __init__(self, X, y, theta, base, link, w=None, aux=None, chunk=4096):
        X = np.asarray(X, dtype=np.float64)
        N, d = X.shape
        S = theta.shape[0]
        self.N, self.d, self.S, self.link = N, d, S, link
        w = np.ones(S) if w is None else np.asarray(w, dtype=np.float64)
        aux = np.ones(S) if aux is None else np.asarray(aux, dtype=np.float64)
        e = np.asarray(base, dtype=np.float64)
        self._data = (X, np.asarray(y, dtype=np.float64), theta, e, w, aux)
        ae, at, aw = np.abs(e), np.abs(theta), np.abs(w)
        self.ll, self.gmu, self.ge = np.zeros(S), np.zeros(d), np.zeros(d)
        # bound = c_z u Wz + c_l u W0 + u Ws: z error, link error, rounding of the sums
        self.Wllz, self.Wll0, self.Wlls = np.zeros(S), np.zeros(S), np.zeros(S)
        self.Wgmuz, self.Wgmu0, self.Wgmus = np.zeros(d), np.zeros(d), np.zeros(d)
        self.Wgez, self.Wge0, self.Wges = np.zeros(d), np.zeros(d), np.zeros(d)
        ns = n_sum(N)
        for lo in range(0, N, chunk):
            Xc, yc = X[lo:lo + chunk], self._data[1][lo:lo + chunk]
            aX = np.abs(Xc)
            ll, r, c, M = link_terms(Xc @ theta.T, yc, link, aux)
            Du = U * (aX @ at.T)                           # z error / c_z
            rw = r * w
            self.ll += ll.sum(axis=0)
            self.gmu += Xc.T @ rw.sum(axis=1)
            self.ge += np.sum(Xc * (rw @ e), axis=0)
            self.Wllz += np.sum(np.abs(r) * Du, axis=0)
            self.Wll0 += np.sum(M, axis=0)
            self.Wlls += ns * np.sum(np.abs(ll), axis=0)
            cz = aw * c * Du                               # |w| c dz / c_z
            r0 = aw * np.abs(r)
            xr = aX.T @ r0.sum(axis=1)
            xre = np.sum(aX * (r0 @ ae), axis=0)
            self.Wgmuz += aX.T @ cz.sum(axis=1)
            self.Wgmu0 += xr
            self.Wgmus += (S + ns) * xr
            self.Wgez += np.sum(aX * (cz @ ae), axis=0)
            self.Wge0 += xre
            self.Wges += (S + ns) * xre

    def bounds(self, c_z=C_Z, c_l=C_L):
        """{'ll' | 'gmu' | 'ge': worst-case bound per element}."""
        return {'ll': c_z * self.Wllz + c_l * U * self.Wll0 + U * self.Wlls,
                'gmu': c_z * self.Wgmuz + c_l * U * self.Wgmu0 + U * self.Wgmus,
                'ge': c_z * self.Wgez + c_l * U * self.Wge0 + U * self.Wges}

    def row(self, n):
        """Contributions of row n to (ll, gmu, ge)."""
        X, y, theta, e, w, aux = self._data
        ll, r, _, _ = link_terms((theta @ X[n])[None, :], y[n:n + 1], self.link, aux)
        rw = (r * w)[0]
        return ll[0], X[n] * rw.sum(), X[n] * (rw @ e)


def ratios(ref, ll, gmu, ge, c_z=C_Z, c_l=C_L):
    """Largest err / bound per output."""
    b = ref.bounds(c_z, c_l)
    out = {}
    for name, got, want in (('ll', ll, ref.ll), ('gmu', gmu, ref.gmu), ('ge', ge, ref.ge)):
        if got is None:
            continue
        err = np.abs(np.asarray(got, dtype=np.float64) - want)
        B = b[name]
        out[name] = float(np.max(np.where(B > 0, err / np.where(B > 0, B, 1.0), np.where(err > 0, np.inf, 0.0))))
    return out


def mutations(ref, bm):
    """The bug classes the element-wise checks must catch, as changes (name, dll, dgmu, dge) of the outputs: a dropped
    row (the last one, the first of the last bm-row tile), a row counted twice, two columns swapped across an 8-column
    group, the largest sample weight lost, a padded sample (theta = e = 0, weight 1) counted, a padded row counted."""
    N, d, S = ref.N, ref.d, ref.S
    X, y, theta, e, w, aux = ref._data
    out = []
    for name, n in (('drop last row', N - 1), ('drop first row of the last tile', (N - 1) // bm * bm)):
        ll, gm, ge = ref.row(n)
        out.append((name, -ll, -gm, -ge))
    ll, gm, ge = ref.row(N // 2)
    out.append(('row counted twice', ll, gm, ge))
    if d >= 2:
        a, b = (7, 8) if d > 8 else (d - 2, d - 1)
        perm = np.arange(d)
        perm[[a, b]] = perm[[b, a]]
        out.append(('columns %d, %d swapped' % (a, b), np.zeros(S), ref.gmu[perm] - ref.gmu, ref.ge[perm] - ref.ge))
    s = int(np.argmax(w))
    sub = Reference(X, y, theta[s:s + 1], e[s:s + 1], ref.link, w=w[s:s + 1], aux=aux[s:s + 1])
    out.append(('weight of sample %d lost' % s, np.zeros(S), -sub.gmu, -sub.ge))
    pad = Reference(X, y, np.zeros((1, d)), np.zeros((1, d)), ref.link)
    out.append(('padded sample counted', np.zeros(S), pad.gmu, pad.ge))
    ll0 = link_terms(np.zeros((1, S)), np.zeros(1) if ref.link == 'gaussian' else np.ones(1), ref.link, aux)[0][0]
    out.append(('padded row counted', ll0, np.zeros(d), np.zeros(d)))
    return out


def detected(ref, dll, dgmu, dge, c_z=C_Z, c_l=C_L):
    """Largest |change| / worst-case bound over every element: > 1 means the element-wise check catches it."""
    b = ref.bounds(c_z, c_l)
    return max(float(np.max(np.abs(dll) / b['ll'])), float(np.max(np.abs(dgmu) / b['gmu'])),
               float(np.max(np.abs(dge) / b['ge'])))


# ---- sweep case shapes: d around every plan regime edge, S around the 16-sample warp chunks and the 256-sample
#      super-chunk, N around the tile height BM and the 148-CTA wave, covered pairwise.  (d, S, N kind)
_CASES = [
    (1, 1, '1'), (1, 257, '2e5'), (1, 16, 'BM+1'), (7, 15, 'BM-1'), (7, 513, 'W+1'), (7, 256, '2e5'),
    (8, 16, 'W-1'), (8, 300, 'BM'), (8, 1, '2e5'), (9, 17, 'BM+1'), (9, 255, '1'), (9, 513, '2e5'),
    (576, 256, 'W+1'), (576, 17, 'BM'), (576, 1, 'W-1'), (576, 15, '2e5'), (577, 300, 'BM-1'), (577, 16, 'W+1'),
    (832, 255, 'W-1'), (832, 15, '1'), (833, 257, 'BM'), (833, 1, 'BM+1'), (864, 513, 'W+1'), (864, 16, 'BM-1'),
    (865, 17, 'W-1'), (865, 300, '1'), (1600, 15, 'BM+1'), (1600, 256, 'W+1'), (1601, 1, 'BM'),
    (1601, 257, 'BM-1'), (2896, 16, 'W+1'), (2896, 255, 'BM+1'), (2896, 513, '1'),
]


def _n(kind, bm):
    return {'1': 1, 'BM-1': bm - 1, 'BM': bm, 'BM+1': bm + 1, 'W-1': 148 * bm - 1, 'W+1': 148 * bm + 1,
            '2e5': 200003}[kind]


CASES = [(_n(k, plan(d)[0]), d, S) for d, S, k in _CASES]


def case_links(N, S):
    """Links run at a case shape: all three where the reference is cheap, else one, rotated by the shape."""
    if N * S <= 2e6:
        return LINKS
    return (LINKS[(N + S) % 3],)


def case_seed(N, d, S):
    return (N * 7919 + d * 31 + S) % (2 ** 31)
