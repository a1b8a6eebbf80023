"""numpy / mpmath references for the streamed LRGaussian log-weights (csrc/lr_stream.cu).

With u = [z, eps] and theta - mu = [B, D] u, log q(theta) needs no solve per draw:
    P = [C^-1 | -C^-1 B^T D^-1],  C C^T = I + B^T D^-2 B,
    log q = -1/2 (d log 2 pi + |u|^2 - |P u|^2) - sum_j log sigma_j + sum_l log P_ll.
`projection` forms P as the kernel's caller must, `log_density_from_base` is the identity, and `mp_log_density` is
the 40-digit value of the Gaussian log density at theta = mu + B z + sigma eps (theta formed in mpmath from the same
base draws), which stays accurate where a float64 dense solve does not (B much larger than sigma)."""
import mpmath
import numpy as np
import scipy.linalg as sla

LOG_2PI = np.log(2.0 * np.pi)


def unpack(vp, d, k):
    vp = np.asarray(vp, dtype=np.float64)
    return vp[:d], vp[d:2 * d], vp[2 * d:].reshape(d, k)


def point(d, k, ratio, rs):
    """var_param with log_sigma ~ 0.1 N(0,1) and B ~ ratio N(0,1): ratio is the scale of B relative to sigma"""
    return np.concatenate([0.3 * rs.randn(d), 0.1 * rs.randn(d), ratio * rs.randn(d * k)])


def projection(vp, d, k):
    """P (k x (k + d)); its left k x k block is the lower-triangular C^-1 with a positive diagonal"""
    _, ls, B = unpack(vp, d, k)
    dinv = np.exp(-ls)
    M = np.eye(k) + (B * (dinv * dinv)[:, None]).T @ B
    C = np.linalg.cholesky(M)
    return np.ascontiguousarray(sla.solve_triangular(C, np.hstack([np.eye(k), -(B * dinv[:, None]).T]), lower=True))


def log_density_from_base(vp, z, eps, P):
    d, k = eps.shape[1], z.shape[1]
    _, ls, _ = unpack(vp, d, k)
    u = np.hstack([z, eps])
    w = u @ P.T
    maha = np.sum(u * u, axis=1) - np.sum(w * w, axis=1)
    return -0.5 * (d * LOG_2PI + maha) - np.sum(ls) + np.sum(np.log(np.diag(P[:, :k])))


def mp_log_density(vp, z, eps, dps=40):
    """log N(mu + B z + sigma eps; mu, B B^T + D^2) in mpmath at `dps` digits, per draw (rows of z, eps)"""
    d, k = eps.shape[1], z.shape[1]
    _, ls, B = unpack(vp, d, k)
    out = []
    with mpmath.workdps(dps):
        sig = [mpmath.exp(mpmath.mpf(float(v))) for v in ls]
        Bm = [[mpmath.mpf(float(B[j, l])) for l in range(k)] for j in range(d)]
        S = mpmath.matrix(d, d)
        for i in range(d):
            for j in range(i + 1):
                v = mpmath.fsum(Bm[i][l] * Bm[j][l] for l in range(k))
                S[i, j] = S[j, i] = v + (sig[i] ** 2 if i == j else 0)
        L = mpmath.cholesky(S)
        logdet = 2 * mpmath.fsum(mpmath.log(L[i, i]) for i in range(d))
        for zr, er in zip(z, eps):
            x = [mpmath.fsum(Bm[j][l] * mpmath.mpf(float(zr[l])) for l in range(k)) + sig[j] * mpmath.mpf(float(er[j]))
                 for j in range(d)]
            y = []
            for i in range(d):                                     # forward substitution L y = x
                y.append((x[i] - mpmath.fsum(L[i, j] * y[j] for j in range(i))) / L[i, i])
            maha = mpmath.fsum(v * v for v in y)
            out.append(float(-(d * mpmath.log(2 * mpmath.pi) + logdet + maha) / 2))
    return np.array(out)
