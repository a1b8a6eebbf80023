"""Variational families -- drop-in mirror of viabel/approximations.py for the in-scope
families (MFGaussian :192-251, MFStudentT :254-312, MultivariateT :322-382).

Sampling and log densities run as CUDA kernels through the C ABI; the O(d) closed forms
(entropy, kl, moments) are evaluated on the host in float64.  Base draws come from a
counter-based Philox generator, not numpy's MT19937 (parity is by draw injection: pass
`base=` to `sample`, or read `last_base` after a call).
"""
from abc import ABC, abstractmethod

import numpy as np
import torch

from . import _lib
from ._tensor import F64, device, is_host, like_input, to_dev

__all__ = ['ApproximationFamily', 'MFGaussian', 'MFStudentT', 'MultivariateT', 'LRGaussian']


class ApproximationFamily(ABC):
    """approximations.py:26-182"""

    def __init__(self, dim, var_param_dim, supports_entropy, supports_kl):
        self._dim = dim
        self._var_param_dim = var_param_dim
        self._supports_entropy = supports_entropy
        self._supports_kl = supports_kl

    def init_param(self):
        return np.zeros(self.var_param_dim)

    @abstractmethod
    def sample(self, var_param, n_samples, seed=None):
        """Generate samples from the variational distribution, shape (n_samples, dim)."""

    def entropy(self, var_param):
        if self.supports_entropy:
            return self._entropy(var_param)
        raise NotImplementedError()

    def _entropy(self, var_param):
        raise NotImplementedError()

    @property
    def supports_entropy(self):
        return self._supports_entropy

    def kl(self, var_param0, var_param1):
        if self.supports_kl:
            return self._kl(var_param0, var_param1)
        raise NotImplementedError()

    def _kl(self, var_param0, var_param1):
        raise NotImplementedError()

    @property
    def supports_kl(self):
        return self._supports_kl

    @abstractmethod
    def log_density(self, var_param, x):
        """Log density of the variational distribution at x."""

    @abstractmethod
    def mean_and_cov(self, var_param):
        """Mean and covariance of the variational distribution."""

    def pth_moment(self, var_param, p):
        if self.supports_pth_moment(p):
            return self._pth_moment(var_param, p)
        raise ValueError('p = {} is not a supported moment'.format(p))

    @abstractmethod
    def _pth_moment(self, var_param, p):
        """pth moment"""

    @abstractmethod
    def supports_pth_moment(self, p):
        """Whether the pth moment is available in closed form."""

    @property
    def dim(self):
        return self._dim

    @property
    def var_param_dim(self):
        return self._var_param_dim


def _host(var_param):
    if isinstance(var_param, torch.Tensor):
        return var_param.detach().cpu().numpy().astype(np.float64)
    return np.asarray(var_param, dtype=np.float64)


class _MeanField(ApproximationFamily):
    """Shared machinery of the two mean-field families; var_param = [mu, log_sigma]."""
    _family = None

    def __init__(self, dim, supports_kl, seed):
        self._seed = int(seed)
        self._offset = 0
        self.quantize_draws = 0          # 1: bf16-exact, 2: fp16-exact draws (exact tensor-core operands)
        self.last_base = None
        super().__init__(dim, 2 * dim, True, supports_kl)

    @property
    def df(self):
        return getattr(self, '_df', float('inf'))

    def init_param(self):
        # approximations.py:207-210, :265-268
        return np.concatenate([np.zeros(self.dim), 2.0 * np.ones(self.dim)])

    # -- base draws ---------------------------------------------------------------------------
    def _draw(self, n, seed, offset):
        raise NotImplementedError

    def stream_length(self, n_samples):
        """Philox stream elements that n_samples draws take: n d normals (or t variates), rounded up to even."""
        n = int(n_samples) * self.dim
        return n + (n & 1)

    def base_draws(self, n_samples, seed=None):
        """Draw (n_samples, dim) base variates on the device.  With seed=None the family's own
        stream advances (like approx._rs); an explicit seed restarts a fresh stream at 0
        (like RandomState(seed), approximations.py:213)."""
        n = int(n_samples) * self.dim
        if seed is None:
            out = self._draw(n, self._seed, self._offset)
            self._offset += self.stream_length(n_samples)
        else:
            out = self._draw(n, int(seed), 0)
        return out.view(int(n_samples), self.dim)

    def sample(self, var_param, n_samples, seed=None, base=None):
        host = is_host(var_param)
        vp = to_dev(var_param)
        if vp.numel() != self.var_param_dim:
            raise ValueError('var_param has the wrong length')
        e = self.base_draws(n_samples, seed) if base is None else to_dev(base)
        self.last_base = e
        theta = torch.empty_like(e)
        _lib.check(_lib.lib.vb_mf_sample_f64(_lib.ptr(vp), _lib.ptr(e), _lib.ptr(theta), e.shape[0],
                                              self.dim, _lib.stream()))
        return like_input(theta, host)

    def log_density(self, var_param, x):
        host = is_host(x)
        vp = to_dev(var_param)
        xd = to_dev(x)
        if xd.dim() == 1:
            xd = xd[None, :]
        out = torch.empty(xd.shape[0], dtype=F64, device=device())
        _lib.check(_lib.lib.vb_mf_log_density_f64(_lib.ptr(vp), _lib.ptr(xd), xd.shape[0], self.dim,
                                                   self._family, float(self.df) if self._family else 0.0,
                                                   _lib.ptr(out), _lib.stream()))
        return like_input(out, host)


class MFGaussian(_MeanField):
    """A mean-field Gaussian approximation family (approximations.py:192-251)."""
    _family = _lib.FAMILY_MF_GAUSSIAN

    def __init__(self, dim, seed=1):
        super().__init__(dim, True, seed)

    def _draw(self, n, seed, offset):
        out = torch.empty(n, dtype=F64, device=device())
        _lib.check(_lib.lib.vb_philox_normal_f64(_lib.ptr(out), n, seed, offset,
                                                  int(self.quantize_draws), _lib.stream()))
        return out

    def _entropy(self, var_param):
        vp = _host(var_param)
        return 0.5 * self.dim * (1.0 + np.log(2 * np.pi)) + np.sum(vp[self.dim:])

    def _kl(self, var_param0, var_param1):
        a, b = _host(var_param0), _host(var_param1)
        d = self.dim
        mean_diff = a[:d] - b[:d]
        dl = a[d:] - b[d:]
        return .5 * np.sum(np.exp(2 * dl) + mean_diff ** 2 / np.exp(2 * b[d:]) - 2 * dl - 1)

    def mean_and_cov(self, var_param):
        vp = _host(var_param)
        return vp[:self.dim].copy(), np.diag(np.exp(2 * vp[self.dim:]))

    def _pth_moment(self, var_param, p):
        v = np.exp(2 * _host(var_param)[self.dim:])
        if p == 2:
            return np.sum(v)
        return 2 * np.sum(v ** 2) + np.sum(v) ** 2

    def supports_pth_moment(self, p):
        return p in [2, 4]


class MFStudentT(_MeanField):
    """A mean-field Student's t approximation family (approximations.py:254-312)."""
    _family = _lib.FAMILY_MF_STUDENT

    def __init__(self, dim, df, seed=1):
        if df <= 2:
            raise ValueError('df must be greater than 2')
        self._df = df
        super().__init__(dim, False, seed)

    def _draw(self, n, seed, offset):
        out = torch.empty(n, dtype=F64, device=device())
        _lib.check(_lib.lib.vb_philox_student_t_f64(_lib.ptr(out), n, float(self._df), seed, offset,
                                                     int(self.quantize_draws), _lib.stream()))
        return out

    def entropy(self, var_param):
        # df-only constants dropped, exactly as approximations.py:276-279
        return np.sum(_host(var_param)[self.dim:])

    def mean_and_cov(self, var_param):
        vp = _host(var_param)
        df = self.df
        return vp[:self.dim].copy(), df / (df - 2) * np.diag(np.exp(2 * vp[self.dim:]))

    def _pth_moment(self, var_param, p):
        df = self.df
        if df <= p:
            raise ValueError('df must be greater than p')
        s2 = np.exp(2 * _host(var_param)[self.dim:])
        c = df / (df - 2)
        if p == 2:
            return c * np.sum(s2)
        return c ** 2 * (2 * (df - 1) / (df - 4) * np.sum(s2 ** 2) + np.sum(s2) ** 2)

    def supports_pth_moment(self, p):
        return p in [2, 4] and p < self.df


class MultivariateT(ApproximationFamily):
    """A full-rank multivariate t approximation family (approximations.py:322-382,
    _distributions.py:7-38).

    var_param = [mu(d), row-major lower triangle of F] with L = tril(F,-1) + diag(exp(diag F)) and
    Sigma = L L^T (paragami PSDSymmetricMatrixPattern, approximations.py:315-319).  Samples use the
    SYMMETRIC square root of Sigma, as the reference does (:348).  The d x d algebra is replicated on every rank.
    Entropy is sum(log L_ii) -- the reference's 0.5*log(det(Sigma)) (:354) overflows for large d (SURVEY.md 7) but is
    the same number.

    Device path (csrc/mvt.cu + csrc/gemm_f64.cu): the Cholesky-vector unpack, Sigma = L L^T, the reparameterisation
    through the eigenbasis and every cotangent GEMM are this package's float64 tensor-core kernels; the symmetric
    eigen-decomposition is the one library call (cuSOLVER via torch.linalg.eigh).

    reparam='cholesky' samples theta = mu + L z / u instead (csrc/mvt_chol.cu).  L L^T = Sigma, so the draws have
    the same distribution and ExclusiveKL / AlphaDivergence are the same functions of var_param, but the gradient is
    a different (equally unbiased) Monte Carlo estimator: per draw it does not match the reference.  Sampling and both
    objectives then cost O(S d^2) float64 tensor-core work with no eigensolver, no d x d temporary and no host
    synchronisation.  Everything else (var_param layout, base draws, log_density, entropy, moments) is the same in
    both modes."""

    REPARAMS = ('sqrtm', 'cholesky')

    def __init__(self, dim, df, seed=1, reparam='sqrtm'):
        if df <= 2:
            raise ValueError('df must be greater than 2')
        if reparam not in self.REPARAMS:
            raise ValueError("reparam must be 'sqrtm' or 'cholesky', got %r" % (reparam,))
        self._reparam = reparam
        self._df = df
        self._seed = int(seed)
        self._offset = 0
        self.last_base = None
        super().__init__(dim, dim + dim * (dim + 1) // 2, True, False)

    @property
    def df(self):
        return self._df

    @property
    def reparam(self):
        """'sqrtm' (theta = mu + (z / u) sqrtm(Sigma), the reference's map) or 'cholesky' (theta = mu + L z / u)."""
        return self._reparam

    def init_param(self):
        # mu = 0, Sigma = 10 I  ->  F = diag(log sqrt(10))   (approximations.py:337-340)
        d = self.dim
        F = np.zeros((d, d))
        F[np.diag_indices(d)] = 0.5 * np.log(10.0)
        return np.concatenate([np.zeros(d), F[np.tril_indices(d)]])

    # -- device pieces (csrc/mvt.cu) ------------------------------------------------------------------
    def unpack(self, vp):
        """(mu[d] view, L[d,d], half_logdet[1] = sum_i F_ii) as CUDA tensors (vb_mvt_unpack_f64)."""
        d = self.dim
        if vp.numel() != self.var_param_dim:
            raise ValueError('var_param has the wrong length')
        L = torch.empty(d, d, dtype=F64, device=vp.device)
        hl = torch.empty(1, dtype=F64, device=vp.device)
        _lib.check(_lib.lib.vb_mvt_unpack_f64(_lib.ptr(vp), d, _lib.ptr(L), _lib.ptr(hl), _lib.stream()))
        return vp[:d], L, hl

    def sigma(self, L, scale=1.0):
        """scale * L L^T through the float64 tensor-core GEMM."""
        d = self.dim
        Sigma = torch.empty(d, d, dtype=F64, device=L.device)
        _lib.check(_lib.lib.vb_mvt_sigma_f64(_lib.ptr(L), d, float(scale), _lib.ptr(Sigma), _lib.stream()))
        return Sigma

    @staticmethod
    def _eigh(Sigma):
        """Symmetric eigendecomposition on the device -- the ONE library call of this path (cuSOLVER through
        torch.linalg.eigh).  cuSOLVER's divide-and-conquer can refuse a large matrix whose eigenvalues are all equal
        (e.g. the reference's init Sigma = 10 I at d = 2048): an exactly diagonal Sigma is then decomposed by sorting
        its diagonal, anything else gets a relative 1e-13 ramp on the diagonal, far below the 1e-10 tolerance.
        Returns (w, V) with V contiguous, eigenvectors in columns."""
        try:
            w, V = torch.linalg.eigh(Sigma)
        except torch.linalg.LinAlgError:
            d = Sigma.shape[0]
            diag = torch.diagonal(Sigma)
            if int(torch.count_nonzero(Sigma)) == int(torch.count_nonzero(diag)):
                # exactly diagonal (the reference's init_param, Sigma = c I): the decomposition is a sort
                w, order = torch.sort(diag)
                V = torch.zeros_like(Sigma)
                V[order, torch.arange(d, device=Sigma.device)] = 1.0
            else:
                ramp = torch.arange(d, dtype=Sigma.dtype, device=Sigma.device) / d
                scale = diag.abs().mean()
                try:
                    w, V = torch.linalg.eigh(Sigma + torch.diag(1e-13 * scale * ramp))
                except torch.linalg.LinAlgError:
                    w, V = torch.linalg.eigh(Sigma + torch.diag(1e-10 * scale * ramp))
        return w.contiguous(), V.contiguous()

    def decompose(self, vp):
        """(L, half_logdet, w, V) of var_param: unpack -> Sigma = L L^T -> eigh."""
        _, L, hl = self.unpack(vp)
        w, V = self._eigh(self.sigma(L))
        return L, hl, w, V

    def transform(self, vp, chi2, z, w, V):
        """(theta[S,d], P[S,d], zu2[S]): theta = mu + (z / u) sqrtm(Sigma) without forming the square root."""
        S, d = int(z.shape[0]), self.dim
        P = torch.empty(S, d, dtype=F64, device=z.device)
        theta = torch.empty(S, d, dtype=F64, device=z.device)
        zu2 = torch.empty(S, dtype=F64, device=z.device)
        ws = torch.empty(_lib.lib.vb_mvt_transform_workspace_bytes(S, d), dtype=torch.uint8, device=z.device)
        _lib.check(_lib.lib.vb_mvt_transform_f64(_lib.ptr(vp), _lib.ptr(z), _lib.ptr(chi2), float(self._df), S, d, _lib.ptr(w),
                                                 _lib.ptr(V), _lib.ptr(P), _lib.ptr(theta), _lib.ptr(zu2), _lib.ptr(ws),
                                                 ws.numel(), _lib.stream()))
        return theta, P, zu2

    def chol_transform(self, vp, chi2, z):
        """(theta[S,d], inv_u[S], zu2[S]): theta = mu + L z / u through the triangular float64 tensor-core kernel
        (vb_mvt_chol_transform_f64), reading L straight from var_param."""
        if vp.numel() != self.var_param_dim:
            raise ValueError('var_param has the wrong length')
        S, d = int(z.shape[0]), self.dim
        if z.dim() != 2 or int(z.shape[1]) != d or chi2.numel() != S:
            raise ValueError('base draws must be chi2[S] and z[S, %d]' % d)
        theta = torch.empty(S, d, dtype=F64, device=z.device)
        inv_u = torch.empty(S, dtype=F64, device=z.device)
        zu2 = torch.empty(S, dtype=F64, device=z.device)
        _lib.check(_lib.lib.vb_mvt_chol_transform_f64(_lib.ptr(vp), _lib.ptr(z), _lib.ptr(chi2), float(self._df), S, d,
                                                      _lib.ptr(theta), _lib.ptr(inv_u), _lib.ptr(zu2), _lib.stream()))
        return theta, inv_u, zu2

    # -- base draws: chi-square FIRST, then normals, as the reference (:345-347) -------------------
    def stream_length(self, n_samples):
        """Philox stream elements that n_samples draws take: n chi-squares, then n d normals, each run rounded up to
        even.  Draw i's chi-square is element i and its normals start at element n + (n & 1) + i d, so a draw can be
        regenerated alone only with the n of the call that drew it."""
        n, d = int(n_samples), self.dim
        return n + (n & 1) + n * d + ((n * d) & 1)

    def base_draws(self, n_samples, seed=None):
        n, d = int(n_samples), self.dim
        dev = device()
        chi2 = torch.empty(n, dtype=F64, device=dev)
        z = torch.empty(n * d, dtype=F64, device=dev)
        s, off = (self._seed, self._offset) if seed is None else (int(seed), 0)
        _lib.check(_lib.lib.vb_philox_chisquare_f64(_lib.ptr(chi2), n, float(self._df), s, off, _lib.stream()))
        off2 = off + n + (n & 1)
        _lib.check(_lib.lib.vb_philox_normal_f64(_lib.ptr(z), n * d, s, off2, 0, _lib.stream()))
        if seed is None:
            self._offset = off + self.stream_length(n)
        return chi2, z.view(n, d)

    def sample(self, var_param, n_samples, seed=None, base=None):
        host = is_host(var_param)
        vp = to_dev(var_param)
        chi2, z = self.base_draws(n_samples, seed) if base is None else (to_dev(base[0]).reshape(-1), to_dev(base[1]))
        self.last_base = (chi2, z)
        if self._reparam == 'cholesky':
            theta, _, _ = self.chol_transform(vp, chi2, z)
        else:
            _, _, w, V = self.decompose(vp)
            theta, _, _ = self.transform(vp, chi2, z, w, V)
        return like_input(theta, host)

    def entropy(self, var_param):
        vp = _host(var_param)
        d = self.dim
        F = np.zeros((d, d))
        F[np.tril_indices(d)] = vp[d:]
        return float(np.sum(np.diag(F)))          # = 0.5 * log det Sigma

    def log_density_device(self, vp, x):
        """multivariate_t_logpdf (_distributions.py:7-38) on CUDA tensors: eigen-decomposition of Sigma,
        eigenvalues <= 1e-10 get a zero inverse but still enter the log pseudo-determinant."""
        d = self.dim
        _, _, w, V = self.decompose(vp)
        x = x.contiguous()
        n = int(x.shape[0])
        out = torch.empty(n, dtype=F64, device=x.device)
        ws = torch.empty(_lib.lib.vb_mvt_log_density_workspace_bytes(n, d), dtype=torch.uint8, device=x.device)
        _lib.check(_lib.lib.vb_mvt_log_density_f64(_lib.ptr(vp), _lib.ptr(w), _lib.ptr(V), _lib.ptr(x), n, d, float(self._df),
                                                   _lib.ptr(out), _lib.ptr(ws), ws.numel(), _lib.stream()))
        return out

    def log_density(self, var_param, x):
        host = is_host(x)
        xd = to_dev(x)
        if xd.dim() == 1:
            xd = xd[None, :]
        return like_input(self.log_density_device(to_dev(var_param), xd), host)

    def mean_and_cov(self, var_param):
        vp = to_dev(var_param)
        mu, L, _ = self.unpack(vp)
        df = self._df
        return mu.cpu().numpy().copy(), self.sigma(L, df / (df - 2.)).cpu().numpy()

    def _pth_moment(self, var_param, p):
        # sums of powers of the eigenvalues of Sigma are traces (approximations.py:364-374 calls eigvalsh):
        # sum lambda = |L|_F^2, sum lambda^2 = |Sigma|_F^2
        df = self._df
        if df <= p:
            raise ValueError('df must be greater than p')
        _, L, _ = self.unpack(to_dev(var_param))
        c = df / (df - 2)
        tr = float((L * L).sum())
        if p == 2:
            return c * tr
        Sigma = self.sigma(L)
        return c ** 2 * (2 * (df - 1) / (df - 4) * float((Sigma * Sigma).sum()) + tr ** 2)

    def supports_pth_moment(self, p):
        return p in [2, 4] and p < self._df


class LRGaussian(ApproximationFamily):
    """A low rank Gaussian approximation family (approximations.py:610-731): Sigma = B B^T + diag(exp(2 log_sigma)),
    var_param = [mu(d), log_sigma(d), B(d,k) row-major] (the PatternDict order of :552-557).  Supports entropy and KL,
    so RAABBVI can run on it.  Everything is evaluated through the k x k capacitance matrix
    M = I + B^T D^-2 B (Woodbury / determinant lemma): O(n d k) for n draws, never a d x d inverse.
    Base draws: z[n,k] FIRST, then eps[n,d] (:641-642), from the family's Philox stream."""

    def __init__(self, dim, seed=1, k=0):
        self._k = int(k)
        self._seed = int(seed)
        self._offset = 0
        self.last_base = None
        super().__init__(dim, 2 * dim + dim * self._k, True, True)

    @property
    def k(self):
        return self._k

    def _normals(self, n, seed, offset):
        out = torch.empty(n, dtype=F64, device=device())
        if n:
            _lib.check(_lib.lib.vb_philox_normal_f64(_lib.ptr(out), n, seed, offset, 0, _lib.stream()))
        return out

    def init_param(self):
        # mu = 0, log_sigma = 1, B ~ N(0,1) from the family's stream (approximations.py:630-634)
        B = self._normals(self.dim * self._k, self._seed, self._offset).cpu().numpy()
        self._offset += B.size + (B.size & 1)
        return np.concatenate([np.zeros(self.dim), np.ones(self.dim), B])

    def unpack(self, vp):
        d, k = self.dim, self._k
        if vp.numel() != self.var_param_dim:
            raise ValueError('var_param has the wrong length')
        return vp[:d], vp[d:2 * d], vp[2 * d:].reshape(d, k)

    def stream_length(self, n_samples):
        """Philox stream elements that n_samples draws take: n k normals for z, then n d for eps, each run rounded up
        to even.  Draw i's z starts at element i k and its eps at n k + ((n k) & 1) + i d, so a draw can be
        regenerated alone only with the n of the call that drew it."""
        n, d, k = int(n_samples), self.dim, self._k
        return n * k + ((n * k) & 1) + n * d + ((n * d) & 1)

    def base_draws(self, n_samples, seed=None):
        n, d, k = int(n_samples), self.dim, self._k
        s, off = (self._seed, self._offset) if seed is None else (int(seed), 0)
        z = self._normals(n * k, s, off).view(n, k)
        off2 = off + n * k + ((n * k) & 1)
        eps = self._normals(n * d, s, off2).view(n, d)
        if seed is None:
            self._offset = off + self.stream_length(n)
        return z, eps

    def sample(self, var_param, n_samples, seed=None, base=None):
        host = is_host(var_param)
        mu, ls, B = self.unpack(to_dev(var_param))
        z, eps = self.base_draws(n_samples, seed) if base is None else (to_dev(base[0]), to_dev(base[1]))
        self.last_base = (z, eps)
        return like_input(mu + z @ B.T + torch.exp(ls) * eps, host)

    # -- Woodbury pieces on torch tensors (differentiable: the objectives reuse them under autograd) --------
    @staticmethod
    def _capacitance(ls, B):
        Dinv2 = torch.exp(-2 * ls)
        M = torch.eye(B.shape[1], dtype=B.dtype, device=B.device) + B.T @ (B * Dinv2[:, None])
        return Dinv2, M

    @classmethod
    def log_det(cls, ls, B):
        """log det(B B^T + D^2) = 2 sum(log_sigma) + log det(I + B^T D^-2 B)   (_get_log_determinant :559-573)."""
        _, M = cls._capacitance(ls, B)
        return 2 * ls.sum() + torch.linalg.slogdet(M)[1]

    @classmethod
    def log_density_t(cls, mu, ls, B, x):
        d = x.shape[1]
        Dinv2, M = cls._capacitance(ls, B)
        diff = x - mu
        t = (diff * Dinv2) @ B                                            # [n, k]
        maha = (diff * diff * Dinv2).sum(dim=1) - (t * torch.linalg.solve(M, t.T).T).sum(dim=1)
        return -0.5 * (d * np.log(2 * np.pi) + 2 * ls.sum() + torch.linalg.slogdet(M)[1] + maha)

    def log_density(self, var_param, x):
        host = is_host(x)
        xd = to_dev(x)
        if xd.dim() == 1:
            xd = xd[None, :]
        mu, ls, B = self.unpack(to_dev(var_param))
        return like_input(self.log_density_t(mu, ls, B, xd), host)

    def _entropy(self, var_param):
        mu, ls, B = self.unpack(to_dev(var_param))
        return float(0.5 * self.dim * (np.log(2 * np.pi) + 1) + 0.5 * self.log_det(ls, B))

    def _kl(self, var_param0, var_param1):
        # 0.5 (log det S1 - log det S0 - d + md^T S1^-1 md + tr(S1^-1 S0))   (:661-687), S1^-1 by Woodbury
        mu0, ls0, B0 = self.unpack(to_dev(var_param0))
        mu1, ls1, B1 = self.unpack(to_dev(var_param1))
        Dinv2, M = self._capacitance(ls1, B1)
        md = mu0 - mu1
        t = (md * Dinv2) @ B1
        maha = (md * md * Dinv2).sum() - t @ torch.linalg.solve(M, t)
        # tr(S1^-1 S0) with S0 = B0 B0^T + D0^2: tr(D1^-2 S0) - tr(M^-1 (B1^T D1^-2) S0 (D1^-2 B1))
        D0sq = torch.exp(2 * ls0)
        W = B1 * Dinv2[:, None]                                           # D1^-2 B1, [d, k]
        tr1 = (Dinv2 * D0sq).sum() + ((B0 * B0) * Dinv2[:, None]).sum()
        WS0W = W.T @ (W * D0sq[:, None]) + (W.T @ B0) @ (B0.T @ W)
        tr2 = torch.trace(torch.linalg.solve(M, WS0W))
        return float(0.5 * (self.log_det(ls1, B1) - self.log_det(ls0, B0) - self.dim + maha + tr1 - tr2))

    def mean_and_cov(self, var_param):
        mu, ls, B = self.unpack(to_dev(var_param))
        return mu.cpu().numpy().copy(), (B @ B.T + torch.diag(torch.exp(2 * ls))).cpu().numpy()

    def _pth_moment(self, var_param, p):
        # sums of eigenvalue powers are traces: sum lambda = tr Sigma, sum lambda^2 = |Sigma|_F^2 (no eigensolver)
        mu, ls, B = self.unpack(to_dev(var_param))
        D2 = torch.exp(2 * ls)
        tr = float(D2.sum() + (B * B).sum())
        if p == 2:
            return tr
        fro2 = float((D2 * D2).sum() + 2 * (D2 * (B * B).sum(dim=1)).sum() + ((B.T @ B) ** 2).sum())
        return 2 * fro2 + tr ** 2

    def supports_pth_moment(self, p):
        return p in [2, 4]
