"""Float64 reference of the tensor-core GLM sweep (vb_glm_fast_sweep, logistic link) and its per-element error model.

With z_ns = y_n x_n.theta_s and r_ns = w_s sigmoid(-z_ns) the sweep returns
    ll[s]  = -sum_n softplus(-z_ns)
    gmu[j] =  sum_n y_n x_nj sum_s r_ns
    ge[j]  =  sum_n y_n x_nj sum_s r_ns e_sj
and, with ll_total_only, the mean over s of ll in every slot.  The reference walks the rows in chunks in float64
(error ~1e-13, far below every budget here).

Error model, per element, from the kernel's numerics (glm_fast.cu):
  GEMM1  fp16 hi/lo split of fp32-cast operands, two correction products on e5m2 copies, fp32 accumulation:
             |dz_ns| <= c_z u_d A_ns,  u_d = 2^-20 + (d/16 + 2) 2^-24,  A_ns = sum_j |y_n x_nj theta_sj|
  E1     MUFU ex2 / lg2 / rcp, ~2^-21 relative; fp32 column sums of 32 rows
  R      stored in fp16: 2^-11 relative plus 2^-25 absolute (subnormal range); rsum (gmu) is fp32, not rounded
  E      stored in fp16: exact for fp16-exact draws, 2^-11 relative otherwise
  E2     x read as X_h + 2^-ax e5m2(X_l 2^ax) (about 2^-14 relative), fp32 sums
Two bounds per element:
  worst-case  W = W0 + c_z Wz            (must never be exceeded)
  statistical T = bias + k sqrt(var)     (roundings are unbiased: k 2^-12 sqrt(sum (x r e)^2) for R and alike; the
                                          roundings of theta and E are shared by all rows and add up coherently over n;
                                          `bias` allows 2^-20 of the absolute sum for the MUFU approximations)
c_z and k are calibrated on a B200 (DESIGN.md 2 lists the largest err / bound ratios measured per output).
"""
import numpy as np

# calibrated constants
C_Z = 8.0
K_STAT = 8.0

LN2 = float(np.log(2.0))
LN2_F32 = float(np.float32(LN2))


def softplus(x):
    return np.logaddexp(0.0, x)


def sigmoid(x):
    return 0.5 * (1.0 + np.tanh(0.5 * x))


def f16_exact(a):
    return np.asarray(a, dtype=np.float64).astype(np.float16).astype(np.float64)


def fp8_scales(X, y):
    """The static power-of-two scales (ax, bx) that vb_glm_fast_create picks for y*X (same formula, host side)."""
    v = (np.asarray(X, dtype=np.float64) * np.asarray(y, dtype=np.float64)[:, None]).astype(np.float32)
    amax = float(np.max(np.abs(v))) if v.size else 0.0
    sumsq = float(np.sum(v.astype(np.float64) ** 2))
    rms = np.sqrt(sumsq / (v.shape[0] * v.shape[1]))
    r = int(np.rint(np.log2(rms))) if rms > 0 else 0
    sexp = int(np.frexp(np.float32(amax))[1]) if amax > 0 else 0
    ax, bx = 2 - r, 8 + r
    ax = min(ax, 26 - sexp)
    bx = max(bx, sexp - 15)
    return ax, bx


def make_case(N, d, S, seed, exact=True):
    """Seeded logistic data with a point theta = beta + e / (2 sqrt(d)): logits of order one, residuals of every size."""
    rs = np.random.RandomState(seed)
    X = rs.randn(N, d)
    beta = rs.randn(d) / np.sqrt(d)
    p = sigmoid(X @ beta)
    y = np.where(rs.rand(N) < p, 1.0, -1.0)
    base = rs.randn(S, d)
    if exact:
        base = f16_exact(base)
    theta = beta + base / (2.0 * np.sqrt(d))
    return X, y, theta, base


def alpha_weights(S, seed):
    """Weights of the shape AlphaDivergence passes (exp(alpha (lw - max lw)), max exactly 1), with exact zeros and
    values down to 1e-30."""
    rs = np.random.RandomState(seed)
    w = np.exp(-rs.exponential(2.0, S))
    w[rs.randint(S)] = 1.0
    if S > 2:
        w[1::7] = 0.0
        w[2::11] = 1e-30
        w[int(np.argmax(w))] = 1.0
    return w


class Reference(object):
    """ll / gmu / ge in float64 and the ingredients of both bounds (c_z and k are applied in `bounds`)."""

    def __init__(self, X, y, theta, base, w=None, exact=True, ax=None, chunk=8192):
        X = np.asarray(X, dtype=np.float64)
        N, d = X.shape
        S = theta.shape[0]
        self.N, self.d, self.S = N, d, S
        w = np.ones(S) if w is None else np.asarray(w, dtype=np.float64)
        self.w = w
        e = np.zeros((S, d)) if base is None else np.asarray(base, dtype=np.float64)
        ae, e2 = np.abs(e), e * e
        at, t2 = np.abs(theta), theta * theta
        u_d = 2.0 ** -20 + (d / 16.0 + 2.0) * 2.0 ** -24
        ax = fp8_scales(X, y)[0] if ax is None else ax
        u_x, floor_x, u_t = 2.0 ** -14, 2.0 ** (-17 - ax), 2.0 ** -13
        u_e = 0.0 if exact else 2.0 ** -11
        self.ll = np.zeros(S)
        self.gmu = np.zeros(d)
        self.ge = np.zeros(d)
        # worst case: W0 + c_z Wz
        self.Wll0, self.Wllz = np.zeros(S), np.zeros(S)
        self.Wgmu0, self.Wgmuz = np.zeros(d), np.zeros(d)
        self.Wge0, self.Wgez = np.zeros(d), np.zeros(d)
        # statistical: bias + k sqrt(Vx + c_z^2 Vz)
        self.Bll, self.Vllz = np.zeros(S), np.zeros(S)
        self.Bgmu, self.Vgmu, self.Vgmuz = np.zeros(d), np.zeros(d), np.zeros(d)
        self.Bge, self.Vge, self.Vgez = np.zeros(d), np.zeros(d), np.zeros(d)
        # the roundings of theta (u_t: its e5m2 low part) and of E are shared by every row: their effects add up
        # coherently over n, through these column sums
        Gs, Gd, Gr = np.zeros((S, d)), np.zeros((S, d)), np.zeros((S, d))
        self._data = (X, y, theta, e, w)
        for lo in range(0, N, chunk):
            Xc = X[lo:lo + chunk] * y[lo:lo + chunk, None]
            aX, X2 = np.abs(Xc), Xc * Xc
            nz = (Xc != 0.0).astype(np.float64)
            z = Xc @ theta.T
            A = aX @ at.T
            Du = u_d * A                                   # worst-case z error / c_z
            eu = u_d * np.sqrt(X2 @ t2.T)                  # typical z error / c_z
            sp = softplus(-z)
            sg = sigmoid(-z)
            dsg = sg * (1.0 - sg)
            r = w * sg
            rb = r.sum(axis=1)
            re = r @ e
            self.ll -= sp.sum(axis=0)
            self.gmu += Xc.T @ rb
            self.ge += np.sum(Xc * re, axis=0)
            self.Wll0 += np.sum(2.0 ** -18 * sp + 2.0 ** -21, axis=0)
            self.Wllz += np.sum(sg * Du, axis=0)
            self.Bll += np.sum(2.0 ** -20 * sp + 2.0 ** -22, axis=0)
            self.Vllz += np.sum((sg * eu) ** 2, axis=0)
            wdz = w * dsg * Du
            wez = w * dsg * eu
            self.Wgmu0 += (u_x + 2.0 ** -16) * (aX.T @ rb) + floor_x * (nz.T @ rb)
            self.Wgmuz += aX.T @ wdz.sum(axis=1)
            self.Bgmu += 2.0 ** -20 * (aX.T @ rb)
            self.Vgmu += (u_x ** 2) * (X2.T @ rb ** 2) + floor_x ** 2 * (nz.T @ rb ** 2)
            self.Vgmuz += X2.T @ (wez ** 2).sum(axis=1)
            rae = r @ ae
            self.Wge0 += (2.0 ** -11 + u_e + 2.0 ** -15 + u_x) * np.sum(aX * rae, axis=0) \
                + 2.0 ** -24 * aX.sum(axis=0) * ae.sum(axis=0) + floor_x * np.sum(nz * np.abs(re), axis=0)
            self.Wgez += np.sum(aX * (wdz @ ae), axis=0)
            self.Bge += 2.0 ** -20 * np.sum(aX * rae, axis=0)
            Gs += sg.T @ Xc
            Gd += (w * dsg).T @ X2
            Gr += r.T @ Xc
            self.Vge += 2.0 ** -24 * np.sum(X2 * ((r * r) @ e2), axis=0) \
                + (u_x ** 2) * np.sum(X2 * re ** 2, axis=0) + floor_x ** 2 * np.sum(nz * re ** 2, axis=0) \
                + 2.0 ** -50 * X2.sum(axis=0) * e2.sum(axis=0)
            self.Vgez += np.sum(X2 * ((wez ** 2) @ e2), axis=0)
        tG = u_t * theta * Gd
        self.Vllc = np.sum((u_t * theta * Gs) ** 2, axis=1)
        self.Vgmuc = np.sum(tG ** 2, axis=0)
        self.Vgec = np.sum((tG * e) ** 2, axis=0) + (u_e / 2.0) ** 2 * np.sum((e * Gr) ** 2, axis=0)

    def row(self, n):
        """Contributions of row n to (ll, gmu, ge)."""
        X, y, theta, e, w = self._data
        x = X[n] * y[n]
        z = theta @ x
        r = w * sigmoid(-z)
        return -softplus(-z), x * r.sum(), x * (r @ e)

    def bounds(self, c_z=C_Z, k=K_STAT):
        """{'ll'|'gmu'|'ge': (worst-case bound, statistical bound)} per element."""
        return {'ll': (self.Wll0 + c_z * self.Wllz, self.Bll + k * np.sqrt(c_z ** 2 * self.Vllz + self.Vllc)),
                'gmu': (self.Wgmu0 + c_z * self.Wgmuz,
                        self.Bgmu + k * np.sqrt(self.Vgmu + c_z ** 2 * self.Vgmuz + self.Vgmuc)),
                'ge': (self.Wge0 + c_z * self.Wgez, self.Bge + k * np.sqrt(self.Vge + c_z ** 2 * self.Vgez + self.Vgec))}

    def total_bound(self, c_z=C_Z):
        """Budget of S * (the ll_total_only mean) against sum_s ll[s]: the per-sample worst cases plus 2^-19 per
        valid row for the fp32 chunk sums that carry the padded columns' ln 2 (subtracted afterwards)."""
        return float(np.sum(self.Wll0 + c_z * self.Wllz)) + 2.0 ** -19 * self.N * max(1, 256 // 64)


def ratios(ref, ll, gmu, ge, c_z=C_Z, k=K_STAT):
    """Largest err / bound per output: {'ll': (worst, stat), ...}."""
    b = ref.bounds(c_z, k)
    out = {}
    for name, got, want in (('ll', ll, ref.ll), ('gmu', gmu, ref.gmu), ('ge', ge, ref.ge)):
        if got is None:
            continue
        err = np.abs(np.asarray(got, dtype=np.float64) - want)
        out[name] = tuple(float(np.max(np.where(B > 0, err / np.where(B > 0, B, 1.0), np.where(err > 0, np.inf, 0.0))))
                          for B in b[name])
    return out


# GPU case shapes: S, d and N around the kernel's branch points (64-sample quarters, 128-sample halves of the e5m2
# Theta copy, 256-column d_pad buckets, 128-row tiles, 256-row super-tiles, 146 -> 148 workspace grid, pairs that run
# one more persistent round than others), covered pairwise.  (N, d, S, general float64 draws?)
CASES = [
    (1, 1, 1, False), (127, 31, 2, False), (128, 255, 63, False), (129, 256, 64, False), (255, 257, 65, True),
    (256, 512, 127, False), (257, 1000, 128, False), (18688, 257, 129, False), (18689, 31, 192, True),
    (38017, 256, 255, False), (129, 2048, 256, False), (257, 1, 255, False), (18689, 512, 256, False),
    (1, 2048, 65, False), (256, 31, 1, False), (38017, 1, 64, False), (127, 1000, 192, True), (255, 2048, 2, False),
    (128, 1, 129, False), (18688, 1000, 63, False),
]


def case_seed(N, d, S):
    return (N * 7919 + d * 31 + S) % (2 ** 31)


def sample_contrib(ref, theta_s, e_s, w_s, chunk=65536):
    """Contributions of one (possibly extra) sample to (gmu, ge), summed over all rows."""
    X, y, _, _, _ = ref._data
    gmu, ge = np.zeros(ref.d), np.zeros(ref.d)
    for lo in range(0, ref.N, chunk):
        Xc = X[lo:lo + chunk] * y[lo:lo + chunk, None]
        r = w_s * sigmoid(-(Xc @ theta_s))
        gmu += Xc.T @ r
        ge += (Xc.T @ r) * e_s
    return gmu, ge


def mutations(ref):
    """The bug classes the element-wise checks are meant to catch, as changes (name, dll, dgmu, dge) of the reference
    outputs: a dropped row (the last one, the first of the last 256-row super-tile, the first), a row counted twice,
    two columns swapped across a 256-column boundary, one sample's weight lost, one padded sample counted."""
    N, d, S = ref.N, ref.d, ref.S
    X, y, theta, e, w = ref._data
    out = []
    last = (N - 1) // 256 * 256
    for name, n in (('drop last row', N - 1), ('drop first row of the last super-tile', last), ('drop row 0', 0)):
        ll, gm, ge = ref.row(n)
        out.append((name, -ll, -gm, -ge))
    ll, gm, ge = ref.row(N // 2)
    out.append(('row counted twice', ll, gm, ge))
    if d >= 2:
        a, b = (255, 256) if d > 256 else (d - 2, d - 1)
        perm = np.arange(d)
        perm[[a, b]] = perm[[b, a]]
        out.append(('columns %d, %d swapped' % (a, b), np.zeros(S), ref.gmu[perm] - ref.gmu, ref.ge[perm] - ref.ge))
    s = int(np.argmax(w))
    gm, ge = sample_contrib(ref, theta[s], e[s], w[s])
    out.append(('weight of sample %d lost' % s, np.zeros(S), -gm, -ge))
    gm, ge = sample_contrib(ref, np.zeros(d), np.zeros(d), 1.0)
    out.append(('padded sample counted', np.zeros(S), gm, ge))
    return out


def detected(ref, dll, dgmu, dge, c_z=C_Z, k=K_STAT):
    """Largest |change| / statistical bound over every element: > 1 means the element-wise check catches it."""
    b = ref.bounds(c_z, k)
    return max(float(np.max(np.abs(dll) / b['ll'][1])), float(np.max(np.abs(dgmu) / b['gmu'][1])),
               float(np.max(np.abs(dge) / b['ge'][1])))
