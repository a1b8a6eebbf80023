"""Model plugin boundary -- mirror of viabel/models.py (Model :11-76) plus the GPU-resident
built-in models named by the north star (logistic / probit regression).

The reference calls user Python under autograd (models.py:27-39).  Here a model either is a
built-in plugin whose S x N likelihood contraction runs as one fused CUDA sweep, or wraps a
user callable on CUDA tensors with an explicit gradient (`Model(log_density, grad)`).
"""
import ctypes

import numpy as np
import torch

from . import _lib
from ._tensor import F64, device, is_host, like_input, to_dev
from .parallel import allreduce_sum_

__all__ = ['Model', 'StanModel', 'GLMModel', 'LogisticRegression', 'ProbitRegression', 'HierarchicalLinearRegression',
           'GaussianTarget', 'StudentTTarget']


class Model(object):
    """Base class for representing a model (models.py:11-76).

    `log_density(theta[S,d]) -> [S]` operates on CUDA float64 tensors.  `grad(theta) -> [S,d]`
    is its gradient; when omitted, torch autograd differentiates `log_density`.
    """

    def __init__(self, log_density, grad=None):
        self._log_density = log_density
        self._grad = grad

    def __call__(self, model_param):
        host = is_host(model_param)
        x = to_dev(model_param)
        squeeze = x.dim() == 1
        if squeeze:
            x = x[None, :]
        out = self._log_density(x)
        if squeeze:
            out = out.reshape(())
        return like_input(out, host)

    def logp_and_grad(self, theta):
        """(log density [S], gradient [S,d]) at CUDA tensor theta[S,d]."""
        if self._grad is not None:
            return self._log_density(theta), self._grad(theta)
        with torch.enable_grad():
            t = theta.detach().requires_grad_(True)
            lp = self._log_density(t)
            (g,) = torch.autograd.grad(lp.sum(), t)
        return lp.detach(), g

    def point_derivatives(self, m, V=None, want_hessian=False):
        """Derivatives of the log density at ONE point m[d] (CUDA tensor), for the control-variate
        ExclusiveKL estimators (objectives.py:200-204, :220-221, :238-239): (grad[d], H V^T as [K,d] or None,
        H[d,d] or None).  Generic models are differentiated by torch autograd (the reference uses autograd's
        grad / make_hvp / hessian); plugins override this with analytic forms."""
        m = m.detach()

        def f(x):
            return self._log_density(x[None, :]).sum()

        with torch.enable_grad():
            x = m.clone().requires_grad_(True)
            (g,) = torch.autograd.grad(f(x), x)
            HV = None
            if V is not None:
                HV = torch.stack([torch.autograd.functional.hvp(f, m, v)[1] for v in V])
            H = torch.autograd.functional.hessian(f, m) if want_hessian else None
        return g.detach(), HV, H

    def constrain(self, model_param):
        raise NotImplementedError()

    @property
    def supports_tempering(self):
        return False

    def set_inverse_temperature(self, inverse_temp):
        raise NotImplementedError()


class StanModel(Model):
    """Adapter for a PyStan fit object (models.py:80-100).  The log density and its gradient are the fit's own
    `log_prob` / `grad_log_prob`, evaluated on the host one row at a time as the reference does
    (`_utils.vectorize_if_needed`): Stan is CPU code and outside the B200 path, so the samples round-trip through host
    memory, while families, objectives, optimisers and diagnostics run on the device as for any `Model(log_density, grad)`."""

    def __init__(self, fit):
        self._fit = fit

        def rows(f, x):
            a = x.detach().cpu().numpy()
            return np.stack([np.asarray(f(r), dtype=np.float64) for r in a])

        super().__init__(lambda x: to_dev(rows(fit.log_prob, x).reshape(-1)),
                         lambda x: to_dev(rows(fit.grad_log_prob, x).reshape(x.shape)))

    def constrain(self, model_param):
        return self._fit.constrain_pars(model_param)


class GLMModel(Model):
    """GPU-resident generalised linear model with an iid N(0, prior_scale^2) prior:

        log p(theta) = sum_n loglik(y_n, x_n . theta) - |theta|^2 / (2 prior_scale^2) + const

    X[N,d] (row-major float64) and y[N] (+1/-1) live in HBM for the lifetime of the object.
    When torch.distributed is initialised and `sharded=True`, X holds this rank's N/world rows
    and the per-sample log-likelihoods and gradient sums are all-reduced (SURVEY.md 8(e)).
    """
    link = None

    def __init__(self, X, y, prior_scale=10.0, sharded=False, process_group=None):
        self.X = to_dev(X)
        self.y = to_dev(y).reshape(-1)
        if self.X.dim() != 2 or self.X.shape[0] != self.y.shape[0]:
            raise ValueError('X must be [N, d] and y must be [N]')
        self.N, self.dim = int(self.X.shape[0]), int(self.X.shape[1])
        self.prior_scale = float(prior_scale)
        self.sharded = bool(sharded)
        self.process_group = process_group
        self._ws = None
        self._ws_S = -1
        self._fast = None          # (handle, model_mem, workspace) of the tensor-core path
        self.path = 'f64'
        super().__init__(self._logp)

    # -- tensor-core fast path ---------------------------------------------------------------------
    @staticmethod
    def _aligned_bytes(nbytes, align=1024):
        buf = torch.empty(nbytes + align, dtype=torch.uint8, device=device())
        off = (-buf.data_ptr()) % align
        return buf[off:off + nbytes]

    def enable_fast_path(self, approx=None):
        """Preprocess the data for the tcgen05 path (fp16 hi+lo split of y*X) and route sweeps of
        up to 256 samples through it.  Raises NotImplementedError when the link or the data range
        is not supported; the float64 path stays available via `path = 'f64'`.

        approx: the variational family that will be fitted on this model.  When given, its base
        draws are switched to fp16-exact values (`approx.quantize_draws = 2`: every N(0,1) / t draw
        is rounded to the nearest float16, a relative perturbation <= 2^-11 of each draw), which
        makes the draws exact tensor-core operands so the back-projection needs one pass instead of
        two.  This changes the sampling distribution in the 4th significant digit of each draw --
        far below Monte Carlo error -- and is the configuration bench.py measures; leave `approx`
        out to keep full-precision draws (they are then rounded inside the kernel only, and the
        fast-path tolerance of 1e-4 still holds)."""
        if approx is not None:
            approx.quantize_draws = 2
        if self._fast is None:
            lib = _lib.lib
            nbytes = lib.vb_glm_fast_model_bytes(self.N, self.dim)
            mem = self._aligned_bytes(nbytes)
            handle = ctypes.c_void_p()
            absmax = ctypes.c_float(0.0)
            _lib.check(lib.vb_glm_fast_create(ctypes.byref(handle), _lib.ptr(self.X), self.X.stride(0),
                                              _lib.ptr(self.y), self.N, self.dim, self.link, _lib.ptr(mem),
                                              mem.numel(), ctypes.byref(absmax), _lib.stream()))
            ws = self._aligned_bytes(lib.vb_glm_fast_workspace_bytes(self.N, self.dim, 256))
            self._fast = (handle, mem, ws)
            self.absmax = absmax.value
        self.path = 'fast'
        return self

    def __del__(self):
        try:
            if self._fast is not None:
                _lib.lib.vb_glm_fast_destroy(self._fast[0])
        except Exception:
            pass

    def _sweep_fast(self, theta, base, w, want_grad, out, debug=None, ll_total_only=False):
        S, d = int(theta.shape[0]), self.dim
        handle, _, ws = self._fast
        ll, gmu, ge = out[:S], out[S:S + d], out[S + d:]
        _lib.check(_lib.lib.vb_glm_fast_sweep(
            handle, _lib.ptr(theta), _lib.ptr(base) if want_grad else None, _lib.ptr(w), S,
            int(bool(want_grad)) | (2 if ll_total_only else 0), _lib.ptr(ll), _lib.ptr(gmu) if want_grad else None,
            _lib.ptr(ge) if want_grad else None, _lib.ptr(ws), ws.numel(), _lib.ptr(debug), _lib.stream()))

    # -- fused sweep -----------------------------------------------------------------------------
    def _workspace(self, S):
        if self._ws_S != S:
            nbytes = _lib.lib.vb_glm_sweep_workspace_bytes(self.N, self.dim, S)
            if nbytes == 0:
                raise NotImplementedError('model dimension too large for the fused sweep')
            self._ws = torch.empty(nbytes, dtype=torch.uint8, device=device())
            self._ws_S = S
        return self._ws

    def _allreduce(self, buf):
        if self.sharded:
            allreduce_sum_(buf, self.process_group)

    def sweep(self, theta, base=None, w=None, want_grad=True, aux=None, ll_total_only=False):
        """One pass over the observations.  Returns (ll[S], gmu[d], ge[d]); the last two are None
        when want_grad is False.  Sums are all-reduced across ranks when sharded.
        ll_total_only: the caller only needs sum_s ll[s] (plain ExclusiveKL value); the fast path
        then skips the per-sample column sums and returns the mean in every ll[s]."""
        S = int(theta.shape[0])
        d = self.dim
        out = torch.empty(S + 2 * d, dtype=F64, device=device())
        ll, gmu, ge = out[:S], out[S:S + d], out[S + d:]
        if self.path == 'fast' and S <= 256 and aux is None:
            self._sweep_fast(theta, base, w, want_grad, out, ll_total_only=ll_total_only)
            if want_grad:
                self._allreduce(out)
                return ll, gmu, ge
            self._allreduce(ll)
            return ll, None, None
        ws = self._workspace(S)
        _lib.check(_lib.lib.vb_glm_sweep_f64(
            _lib.ptr(self.X), self.X.stride(0), _lib.ptr(self.y), self.N, d, self.link,
            _lib.ptr(theta), _lib.ptr(base) if want_grad else None, _lib.ptr(w), _lib.ptr(aux), S,
            int(bool(want_grad)), _lib.ptr(ll), _lib.ptr(gmu) if want_grad else None,
            _lib.ptr(ge) if want_grad else None, _lib.ptr(ws), ws.numel(), _lib.stream()))
        if want_grad:
            self._allreduce(out)
            return ll, gmu, ge
        self._allreduce(ll)
        return ll, None, None

    def logp_and_grad(self, theta, chunk=65536):
        """Per-sample log density [S] and gradient [S,d] (needed by full-rank / low-rank / flow families, whose
        cotangents use every sample's gradient).  The S x d accumulator does not fit on chip, so this is two GEMMs on
        the package's float64 DMMA kernel (vb_gemm_f64: A = y.(X_c Theta^T) with the row scaling fused, then
        G += A^T X_c) with the link step between them (vb_glm_link_f64), over row chunks; the fused sweep above is
        the mean-field hot path."""
        theta = theta.contiguous()
        S, d = int(theta.shape[0]), int(theta.shape[1])
        lib, ptr, st = _lib.lib, _lib.ptr, _lib.stream()
        ll = torch.zeros(S, dtype=F64, device=theta.device)
        G = torch.zeros_like(theta)
        rows = min(int(chunk), self.N)
        A = torch.empty(rows, S, dtype=F64, device=theta.device)
        Gc = torch.empty_like(theta)
        ws = torch.empty(max(8, lib.vb_glm_link_workspace_bytes(rows, S)), dtype=torch.uint8, device=theta.device)
        ldx = self.X.stride(0)
        for lo in range(0, self.N, rows):
            nc = min(rows, self.N - lo)
            Xc, yc = self.X[lo:lo + nc], self.y[lo:lo + nc]
            _lib.check(lib.vb_gemm_f64(0, 1, nc, S, d, 1.0, ptr(Xc), ldx, ptr(theta), d, ptr(A), S, None, ptr(yc), None, None,
                                       None, st))
            _lib.check(lib.vb_glm_link_f64(ptr(A), ptr(yc), nc, S, self.link, ptr(ll), ptr(ws), ws.numel(), st))
            _lib.check(lib.vb_gemm_f64(1, 0, S, d, nc, 1.0, ptr(A), S, ptr(Xc), ldx, ptr(Gc), d, None, None, None, None, None, st))
            G += Gc
        buf = torch.cat([ll, G.reshape(-1)])
        self._allreduce(buf)
        ll, G = buf[:S], buf[S:].view_as(theta)
        return ll + self.log_prior(theta), G - theta / self.prior_scale ** 2

    def point_derivatives(self, m, V=None, want_hessian=False):
        """Model.point_derivatives through vb_glm_point_f64: gradient and up to 8 Hessian-vector products in one
        pass over X, the full Hessian as a weighted SYRK on the FP64 tensor pipe; the prior's part added here.
        Sums are all-reduced when the observations are sharded."""
        d = self.dim
        m = m.detach().to(F64).contiguous()
        K = 0 if V is None else int(V.shape[0])
        if K > 8:
            parts = [self.point_derivatives(m, V[i:i + 8], False)[1] for i in range(0, K, 8)]
            g, _, H = self.point_derivatives(m, None, want_hessian)
            return g, torch.cat(parts), H
        Kp = K if K <= 4 else 8
        Vp = None
        if K:
            Vp = torch.zeros(Kp, d, dtype=F64, device=m.device)
            Vp[:K] = V
        nbytes = _lib.lib.vb_glm_point_workspace_bytes(self.N, d, Kp, int(want_hessian))
        ws = torch.empty(max(nbytes, 8), dtype=torch.uint8, device=m.device)
        n_out = d + Kp * d + (d * d if want_hessian else 0)
        out = torch.zeros(n_out, dtype=F64, device=m.device)
        g, HV = out[:d], out[d:d + Kp * d].view(Kp, d) if Kp else None
        H = out[d + Kp * d:].view(d, d) if want_hessian else None
        _lib.check(_lib.lib.vb_glm_point_f64(
            _lib.ptr(self.X), self.X.stride(0), _lib.ptr(self.y), self.N, d, self.link, _lib.ptr(m), _lib.ptr(Vp), Kp,
            None, _lib.ptr(g), _lib.ptr(HV) if Kp else None, _lib.ptr(H) if want_hessian else None,
            _lib.ptr(ws), ws.numel(), _lib.stream()))
        self._allreduce(out)
        it2 = 1.0 / self.prior_scale ** 2
        g = g - m * it2
        if K:
            HV = HV[:K] - V * it2
        else:
            HV = None
        if want_hessian:
            H = H - it2 * torch.eye(d, dtype=F64, device=m.device)
        return g, HV, H

    def log_prior(self, theta):
        d = self.dim
        return (-0.5 * (theta * theta).sum(dim=1) / self.prior_scale ** 2
                - d * np.log(self.prior_scale * np.sqrt(2 * np.pi)))

    def _logp(self, theta):
        ll, _, _ = self.sweep(theta.contiguous(), want_grad=False)
        return ll + self.log_prior(theta)


class LogisticRegression(GLMModel):
    """Bayesian logistic regression, y in {-1,+1} (BASELINE.json configs 1-3)."""
    link = _lib.LINK_LOGISTIC


class ProbitRegression(GLMModel):
    """Bayesian probit regression, y in {-1,+1}."""
    link = _lib.LINK_PROBIT


class HierarchicalLinearRegression(Model):
    """GPU-resident hierarchical linear regression (BASELINE.json configs[3], SURVEY.md 8(d) C4):

        y_i ~ N(x_i . beta_{g(i)}, sigma),  beta_g ~ N(m, tau I),  m ~ N(0, 10 I),
        log tau ~ N(0,1),  log sigma ~ N(0,1);   theta = [beta (G*p, group-major), m (p), log tau, log sigma].

    Log density and PER-SAMPLE gradients (what the full-rank families need) through vb_hier_logp_grad_f64: the
    observations are kept sorted by group and the likelihood is a grouped contraction -- one CTA per (group, 128
    samples) -- not a dense GEMM against a block-expanded [N, G*p] design matrix."""

    def __init__(self, X, y, group, n_groups):
        Xd = to_dev(X)
        yd = to_dev(y).reshape(-1)
        g = torch.as_tensor(np.asarray(group), dtype=torch.int64, device=Xd.device)
        self.N, self.p = int(Xd.shape[0]), int(Xd.shape[1])
        self.G = int(n_groups)
        if self.p > 32:
            raise NotImplementedError('at most 32 coefficients per group')
        self.dim = self.G * self.p + self.p + 2
        order = torch.argsort(g, stable=True)
        self.X = Xd[order].contiguous()
        self.y = yd[order].contiguous()
        counts = torch.bincount(g, minlength=self.G)
        self.goff = torch.cat([torch.zeros(1, dtype=torch.int64, device=Xd.device), torch.cumsum(counts, 0)]).contiguous()
        super().__init__(lambda th: self.logp_and_grad(th, want_grad=False)[0], lambda th: self.logp_and_grad(th)[1])

    def logp_and_grad(self, theta, want_grad=True):
        theta = theta.contiguous()
        S = int(theta.shape[0])
        if theta.shape[1] != self.dim:
            raise ValueError('theta must be [S, %d]' % self.dim)
        lp = torch.empty(S, dtype=F64, device=theta.device)
        grad = torch.empty(S, self.dim, dtype=F64, device=theta.device) if want_grad else None
        ws = torch.empty(_lib.lib.vb_hier_workspace_bytes(self.G, S), dtype=torch.uint8, device=theta.device)
        _lib.check(_lib.lib.vb_hier_logp_grad_f64(_lib.ptr(self.X), _lib.ptr(self.y), _lib.ptr(self.goff), self.N, self.p,
                                                  self.G, _lib.ptr(theta), S, _lib.ptr(lp), _lib.ptr(grad), _lib.ptr(ws),
                                                  ws.numel(), _lib.stream()))
        return lp, grad


def _target_logp_grad(theta, kind, loc, scale, df, const):
    """(log p[S], grad[S,d]) of a product target through vb_target_logp_grad_f64 (csrc/targets.cu)."""
    th = theta.contiguous()
    if th.dim() == 1:
        th = th[None, :]
    S, d = int(th.shape[0]), int(th.shape[1])
    if d != loc.numel():
        raise ValueError('theta has the wrong dimension')
    lp = torch.empty(S, dtype=F64, device=th.device)
    G = torch.empty(S, d, dtype=F64, device=th.device)
    _lib.check(_lib.lib.vb_target_logp_grad_f64(_lib.ptr(th), S, d, kind, _lib.ptr(loc), _lib.ptr(scale), float(df),
                                               float(const), _lib.ptr(lp), _lib.ptr(G), _lib.stream()))
    return lp, G


def _product_target(model):
    """(kind, loc, scale, df) of a built-in product target for the fused kernels, else None (exact types only)."""
    if type(model) in (GaussianTarget, StudentTTarget):
        return (0, model.mean, model.sd, 0.0) if type(model) is GaussianTarget else (1, model.loc, model.scale, model.df)
    return None


class GaussianTarget(Model):
    """Independent Gaussian target sum_j N(theta_j; mean_j, sd_j) (the reference tests' target,
    tests/test_objectives.py:18-19) with its analytic gradient."""

    def __init__(self, mean, sd):
        self.mean, self.sd = to_dev(mean).reshape(-1), to_dev(sd).reshape(-1)
        self.dim = int(self.mean.numel())
        self._const = float(-(torch.log(self.sd).sum() + 0.5 * self.dim * np.log(2 * np.pi)))
        super().__init__(lambda th: self.logp_and_grad(th)[0], lambda th: self.logp_and_grad(th)[1])

    def logp_and_grad(self, theta):
        return _target_logp_grad(theta, 0, self.mean, self.sd, 0.0, self._const)

    def point_derivatives(self, m, V=None, want_hessian=False):
        h = -1.0 / (self.sd * self.sd)                    # diagonal Hessian
        g = -(m - self.mean) / (self.sd * self.sd)
        return g, None if V is None else V * h, torch.diag(h) if want_hessian else None


class StudentTTarget(Model):
    """Product Student-t target sum_j t_df(theta_j; loc_j, scale_j) (SURVEY.md 8(d) C5)."""

    def __init__(self, loc, scale, df):
        import math
        self.loc, self.scale, self.df = to_dev(loc).reshape(-1), to_dev(scale).reshape(-1), float(df)
        self.dim = int(self.loc.numel())
        df = self.df
        self._const = self.dim * (math.lgamma(0.5 * (df + 1)) - math.lgamma(0.5 * df) - 0.5 * math.log(df * math.pi)) \
            - float(torch.log(self.scale).sum())
        super().__init__(lambda th: self.logp_and_grad(th)[0], lambda th: self.logp_and_grad(th)[1])

    def logp_and_grad(self, theta):
        return _target_logp_grad(theta, 1, self.loc, self.scale, self.df, self._const)

    def point_derivatives(self, m, V=None, want_hessian=False):
        df = self.df
        z = (m - self.loc) / self.scale
        g = -(df + 1.0) * z / ((df + z * z) * self.scale)
        h = -(df + 1.0) * (df - z * z) / ((df + z * z) ** 2 * self.scale * self.scale)
        return g, None if V is None else V * h, torch.diag(h) if want_hessian else None
