"""Variational objectives -- drop-in mirror of viabel/objectives.py for the hot path:
ExclusiveKL (:108-168, entropy and path-derivative forms) and AlphaDivergence (:419-463).

The reference differentiates a Python closure with autograd; here `objective(var_param)`
launches the fused CUDA sweep (sample -> model log density + gradient -> reduction) and
assembles the analytic gradient of SURVEY.md App. A on the device.
"""
import math
from abc import ABC, abstractmethod

import numpy as np
import torch

from . import _lib
from ._tensor import F64, device, is_host, to_dev
from .approximations import LRGaussian, MultivariateT, _MeanField
from .flows import NVPFlow
from .models import GLMModel, Model
from .parallel import broadcast_seed, is_distributed

__all__ = ['VariationalObjective', 'StochasticVariationalObjective', 'ExclusiveKL', 'AlphaDivergence',
           'DISInclusiveKL']


class VariationalObjective(ABC):
    """A variational objective to minimise (objectives.py:17-79)."""

    def __init__(self, approx, model):
        self._approx = approx
        self._model = model if isinstance(model, Model) or model is None else Model(model)
        self._objective_and_grad = None
        self._update_objective_and_grad()

    def __call__(self, var_param):
        if self._objective_and_grad is None:
            raise RuntimeError("no objective and gradient available")
        return self._objective_and_grad(var_param)

    @abstractmethod
    def _update_objective_and_grad(self):
        """Rebuild the objective when approx / model / num_mc_samples change."""

    def update(self, var_param, direction):
        """objectives.py:57-59"""
        return var_param - direction

    @property
    def approx(self):
        return self._approx

    @approx.setter
    def approx(self, value):
        self._approx = value
        self._update_objective_and_grad()

    @property
    def model(self):
        return self._model

    @model.setter
    def model(self, value):
        self._model = value if isinstance(value, Model) else Model(value)
        self._update_objective_and_grad()


class StochasticVariationalObjective(VariationalObjective):
    """objectives.py:82-105"""

    def __init__(self, approx, model, num_mc_samples):
        self._num_mc_samples = num_mc_samples
        super().__init__(approx, model)

    @property
    def num_mc_samples(self):
        return self._num_mc_samples

    @num_mc_samples.setter
    def num_mc_samples(self, value):
        self._num_mc_samples = value
        self._update_objective_and_grad()


def _workspace(lib_fn_entropy, lib_fn_path, objective, S, d, device):
    nbytes = (lib_fn_path if objective == _lib.OBJ_EXCLUSIVE_KL_PATH else lib_fn_entropy)(S, d)
    return torch.empty(nbytes, dtype=torch.uint8, device=device)


def _mvt_objective(approx, model, S, objective, alpha, var_param, base=None, seed=None):
    """ExclusiveKL (entropy and path-derivative branches) / AlphaDivergence for the full-rank MultivariateT family
    (objectives.py:154-164, :443-460 with approximations.py:342-357; gradient per SURVEY.md App. A.3).
    unpack -> Sigma -> [cuSOLVER eigh] -> reparameterise -> model plugin -> vb_mvt_objective_f64: everything except
    the eigensolver is this package's kernels (csrc/mvt.cu, float64 tensor-core GEMMs of csrc/gemm_f64.cu)."""
    vp = to_dev(var_param)
    d, df = approx.dim, float(approx.df)
    chi2, z = approx.base_draws(S, seed) if base is None else (to_dev(base[0]).reshape(-1), to_dev(base[1]))
    approx.last_base = (chi2, z)
    S = int(z.shape[0])
    if approx.reparam == 'cholesky':
        return _mvt_chol_objective(approx, model, objective, alpha, vp, chi2, z)
    L, hl, w, V = approx.decompose(vp)
    theta, P, zu2 = approx.transform(vp, chi2, z, w, V)
    f, G = model.logp_and_grad(theta)
    out = torch.empty(1 + vp.numel(), dtype=F64, device=vp.device)
    ws = _workspace(_lib.lib.vb_mvt_objective_workspace_bytes, _lib.lib.vb_mvt_path_workspace_bytes, objective, S, d,
                    vp.device)
    _lib.check(_lib.lib.vb_mvt_objective_f64(
        _lib.ptr(L), _lib.ptr(hl), _lib.ptr(w), _lib.ptr(V), _lib.ptr(P), _lib.ptr(zu2), _lib.ptr(f.contiguous()),
        _lib.ptr(G.contiguous()), S, d, df, objective, float(alpha), _lib.ptr(out[:1]), _lib.ptr(out[1:]), _lib.ptr(ws),
        ws.numel(), _lib.stream()))
    return out[0], out[1:]


def _mvt_chol_objective(approx, model, objective, alpha, vp, chi2, z):
    """The same objectives in MultivariateT's Cholesky reparameterisation, theta = mu + L z / u: triangular transform
    -> model plugin -> vb_mvt_chol_objective_f64 (csrc/mvt_chol.cu).  No eigensolver and no host synchronisation.
    The path-derivative form inverts L on the device and needs an O(d^2 + S d) workspace; the others need O(S)."""
    S, d = int(z.shape[0]), approx.dim
    theta, inv_u, zu2 = approx.chol_transform(vp, chi2, z)
    f, G = model.logp_and_grad(theta)
    out = torch.empty(1 + vp.numel(), dtype=F64, device=vp.device)
    ws = _workspace(_lib.lib.vb_mvt_chol_objective_workspace_bytes, _lib.lib.vb_mvt_chol_path_workspace_bytes, objective,
                    S, d, vp.device)
    _lib.check(_lib.lib.vb_mvt_chol_objective_f64(
        _lib.ptr(vp), _lib.ptr(z), _lib.ptr(inv_u), _lib.ptr(zu2), _lib.ptr(f.contiguous()), _lib.ptr(G.contiguous()), S, d,
        float(approx.df), objective, float(alpha), _lib.ptr(out[:1]), _lib.ptr(out[1:]), _lib.ptr(ws), ws.numel(),
        _lib.stream()))
    return out[0], out[1:]


class _ModelLogDensity(torch.autograd.Function):
    """f(theta) with the model plugin's own gradient kernels as the backward pass (no autograd inside the model)."""

    @staticmethod
    def forward(ctx, theta, model):
        f, G = model.logp_and_grad(theta.detach().contiguous())
        ctx.save_for_backward(G)
        return f

    @staticmethod
    def backward(ctx, grad_out):
        (G,) = ctx.saved_tensors
        return grad_out[:, None] * G, None


def _lr_objective(approx, model, S, objective, alpha, var_param, base=None, seed=None):
    """ExclusiveKL (entropy / path-derivative) and AlphaDivergence for LRGaussian (objectives.py:154-164, :443-460 with
    approximations.py:638-646).  The model's log density and gradient come from the plugin's kernels; the O(S d k)
    reparameterisation and the k x k Woodbury algebra of log q / entropy are differentiated by torch autograd."""
    vp = to_dev(var_param)
    z, eps = approx.base_draws(S, seed) if base is None else (to_dev(base[0]), to_dev(base[1]))
    approx.last_base = (z, eps)
    S = eps.shape[0]
    d = approx.dim
    with torch.enable_grad():
        lam = vp.detach().clone().requires_grad_(True)
        mu, ls, B = approx.unpack(lam)
        theta = mu + z @ B.T + torch.exp(ls) * eps
        f = _ModelLogDensity.apply(theta, model)
        if objective == _lib.OBJ_EXCLUSIVE_KL:
            value = -(f.mean() + 0.5 * d * (np.log(2 * np.pi) + 1) + 0.5 * approx.log_det(ls, B))
        elif objective == _lib.OBJ_EXCLUSIVE_KL_PATH:
            mu0, ls0, B0 = approx.unpack(vp.detach())
            value = -(f - approx.log_density_t(mu0, ls0, B0, theta)).mean()
        else:
            lw = f - approx.log_density_t(mu, ls, B, theta)
            m = lw.max().detach()
            sv = torch.exp(lw - m) ** alpha
            # the reference's gradient is alpha * mean(sv.detach() * d lw) -- NOT divided by mean(sv) (SURVEY App. A.2)
            surrogate = alpha * (sv.detach() * lw).mean()
            (grad,) = torch.autograd.grad(surrogate, lam)
            return (torch.log(sv.mean()) / alpha + m).detach(), grad
        (grad,) = torch.autograd.grad(value, lam)
    return value.detach(), grad


def _flow_objective(approx, model, S, objective, alpha, var_param, base=None, seed=None):
    """ExclusiveKL (path-derivative form) and AlphaDivergence for NVPFlow (objectives.py:154-164, :443-460 with
    approximations.py:493-539).  z_0 comes from the prior's Philox stream (or `base`: the prior's base draws), the
    coupling networks and the prior's log density are differentiated by torch autograd, the model's log density and
    gradient come from the plugin.  The family has no entropy, and the reference's plain ExclusiveKL branch cannot
    evaluate it either (it calls approx.log_density(samples) without var_param, objectives.py:163 -> TypeError)."""
    if objective == _lib.OBJ_EXCLUSIVE_KL:
        raise NotImplementedError('NVPFlow has no entropy: use ExclusiveKL(..., use_path_deriv=True) or AlphaDivergence '
                                  '(the reference raises a TypeError on this branch, objectives.py:163)')
    vp = to_dev(var_param)
    z0 = approx.prior_draws(S, seed=seed, base=base)
    with torch.enable_grad():
        lam = vp.detach().clone().requires_grad_(True)
        x = approx.g_t(lam, z0)
        f = _ModelLogDensity.apply(x, model)
        if objective == _lib.OBJ_EXCLUSIVE_KL_PATH:
            value = -(f - approx.log_density_t(vp.detach(), x)).mean()
            (grad,) = torch.autograd.grad(value, lam)
            return value.detach(), grad
        lw = f - approx.log_density_t(lam, x)
        m = lw.max().detach()
        sv = torch.exp(lw - m) ** alpha
        surrogate = alpha * (sv.detach() * lw).mean()                  # unnormalised, as the reference (App. A.2)
        (grad,) = torch.autograd.grad(surrogate, lam)
        approx.last_log_weights = lw.detach()
        return (torch.log(sv.mean()) / alpha + m).detach(), grad


def _to_host(value, grad):
    """(value, grad) -> (float, numpy) with ONE device-to-host copy when both are views of the same
    [1 + len(grad)] buffer (the layout _mf_objective produces), else one copy each."""
    base = grad._base
    if base is not None and base is value._base and base.dim() == 1 and base.numel() == grad.numel() + 1:
        h = base.cpu().numpy()
        return float(h[0]), h[1:].copy()
    return float(value), grad.cpu().numpy()


def _mf_objective(approx, model, S, objective, alpha, var_param, base=None, seed=None, want_logp=False):
    """One fused evaluation for a mean-field family.  Returns (value, grad[, logp]) as 0-d / 1-d
    CUDA tensors (no host sync)."""
    if isinstance(approx, MultivariateT):
        return _mvt_objective(approx, model, S, objective, alpha, var_param, base=base, seed=seed)
    if isinstance(approx, LRGaussian):
        return _lr_objective(approx, model, S, objective, alpha, var_param, base=base, seed=seed)
    if isinstance(approx, NVPFlow):
        return _flow_objective(approx, model, S, objective, alpha, var_param, base=base, seed=seed)
    if not isinstance(approx, _MeanField):
        raise NotImplementedError('only mean-field families are supported by this objective path')
    d = approx.dim
    vp = to_dev(var_param)
    if vp.numel() != 2 * d:
        raise ValueError('var_param has the wrong length')
    e = approx.base_draws(S, seed) if base is None else to_dev(base)
    approx.last_base = e
    S = int(e.shape[0])
    dev = device()
    theta = torch.empty_like(e)
    lib, ptr, st = _lib.lib, _lib.ptr, _lib.stream()
    _lib.check(lib.vb_mf_sample_f64(ptr(vp), ptr(e), ptr(theta), S, d, st))
    family, df = approx._family, float(approx.df) if approx._family else 0.0
    out = torch.empty(1 + 2 * d, dtype=F64, device=dev)
    value, grad = out[:1], out[1:]
    logp = torch.empty(S, dtype=F64, device=dev) if want_logp else None
    glm = isinstance(model, GLMModel)
    prior_sd = model.prior_scale if glm else float('inf')

    def sweep(w):
        if glm:
            # plain ExclusiveKL only needs mean_s ll[s]; per-sample values are kept when asked for
            total_only = objective == _lib.OBJ_EXCLUSIVE_KL and not want_logp
            return model.sweep(theta, e, w, True, ll_total_only=total_only)
        f, G = model.logp_and_grad(theta)
        G = G.to(F64).contiguous()
        gv = torch.empty(2 * d, dtype=F64, device=dev)
        _lib.check(lib.vb_mf_reduce_grads_f64(ptr(G), ptr(w), ptr(e), S, d, ptr(gv[:d]), ptr(gv[d:]), st))
        return f.contiguous(), gv[:d], gv[d:]

    w = None
    if objective == _lib.OBJ_ALPHA:
        if glm:
            ll, _, _ = model.sweep(theta, None, None, False)
        else:
            ll = model.logp_and_grad(theta)[0].contiguous()
        lw = torch.empty(S, dtype=F64, device=dev)
        w = torch.empty(S, dtype=F64, device=dev)
        _lib.check(lib.vb_mf_alpha_weights_f64(ptr(vp), ptr(theta), ptr(e), ptr(ll), S, d, family, df,
                                               prior_sd, float(alpha), ptr(lw), ptr(w), ptr(value), st))
        approx.last_log_weights = lw            # log p - log q per sample (objectives.py:446)
    ll, gmu, ge = sweep(w)
    ws = torch.empty(max(8, lib.vb_mf_objective_finish_workspace_bytes(S)), dtype=torch.uint8, device=dev)
    _lib.check(lib.vb_mf_objective_finish_f64(
        ptr(vp), ptr(theta), ptr(e), ptr(ll), ptr(gmu), ptr(ge), ptr(w), S, d, family, df, prior_sd,
        objective, float(alpha), ptr(value), ptr(grad), ptr(logp), ptr(ws), ws.numel(), st))
    if want_logp:
        return value[0], grad, logp
    return value[0], grad


class ExclusiveKL(StochasticVariationalObjective):
    """Exclusive KL / negative ELBO with the reparameterised gradient (objectives.py:108-168)."""

    def __init__(self, approx, model, num_mc_samples, use_path_deriv=False, hessian_approx_method=None):
        self._use_path_deriv = use_path_deriv
        if hessian_approx_method in [None, 'full', 'mean_only', 'loo_diag_approx', 'loo_direct_approx']:
            self.hessian_approx_method = hessian_approx_method
        else:
            raise ValueError("Name of approximation must be one of 'full', 'mean_only', 'loo_diag_approx', 'loo_direct_approx' or None object.")
        super().__init__(approx, model, num_mc_samples)

    def _control_variate_objective(self, var_param, base=None):
        """ExclusiveKL with the control-variate gradient estimators of objectives.py:170-273 (after Miller et al.,
        "Reducing Reparameterization Gradient Variance").

        The reference forms per-sample control variates from the model's gradient g_m and Hessian H at the
        variational mean m and averages them.  Averaged over the S samples (u_s = z_s - m, ubar = mean_s u_s,
        T_j = mean_s u_sj (H u_s)_j) every estimator collapses to the plain reparameterisation gradient plus

            mean part   : + H ubar                                       (all four methods)
            scale part  : full             : + g_m * ubar + T - diag(H) * s^2
                          loo_diag_approx  : + g_m * ubar     (the leave-one-out diagonals cancel in the mean)
                          mean_only, loo_direct_approx : nothing

        so one evaluation costs the usual fused sweep plus ONE extra pass over the data (vb_glm_point_f64:
        gradient and a single Hessian-vector product at m), or the weighted-SYRK Hessian for 'full'.  Identical to
        the per-sample formulas to rounding (tests/golden/objectives_cv.npz, generated by the reference)."""
        approx, model = self.approx, self.model
        if not isinstance(approx, _MeanField):
            raise NotImplementedError('control-variate estimators are implemented for mean-field families')
        host = is_host(var_param)
        vp = to_dev(var_param)
        d, S = approx.dim, self.num_mc_samples
        # plain reparameterisation estimate: the reference's g_hat_rprm_grad (objectives.py:192-198) is the
        # entropy-form gradient whichever way the value is computed
        value, grad = _mf_objective(approx, model, S, _lib.OBJ_EXCLUSIVE_KL, 0.0, vp, base=base)
        e = approx.last_base
        S = int(e.shape[0])
        mu, ls = vp[:d], vp[d:]
        sig = torch.exp(ls)
        if self._use_path_deriv:
            # value = -mean(f - log q) = entropy-form value + H(q) + mean_s log q(z_s)      (objectives.py:176-180)
            theta = torch.empty_like(e)
            _lib.check(_lib.lib.vb_mf_sample_f64(_lib.ptr(vp), _lib.ptr(e), _lib.ptr(theta), S, d, _lib.stream()))
            logq = approx.log_density(vp, theta)
            value = value + float(approx.entropy(vp)) + logq.mean()
        # ubar = mean_s (z_s - m) = sigma * mean_s e_s: column means through the sample-moments kernel
        ebar = torch.empty(d, dtype=F64, device=vp.device)
        ws = torch.empty(max(8, _lib.lib.vb_sample_moments_workspace_bytes(S, d, 0)), dtype=torch.uint8, device=vp.device)
        _lib.check(_lib.lib.vb_sample_moments_f64(_lib.ptr(e), S, d, d, _lib.ptr(ebar), None, None, None, _lib.ptr(ws),
                                                  ws.numel(), _lib.stream()))
        ubar = sig * ebar
        method = self.hessian_approx_method
        g_m, HV, H = model.point_derivatives(mu, ubar[None, :], want_hessian=(method == 'full'))
        corr = torch.zeros_like(grad)
        corr[:d] = HV[0]
        if method == 'full':
            U = sig * e                                                   # z_s - m
            T = (U * (U @ H)).mean(dim=0)                                 # library GEMM, S x d x d
            scale2 = sig * sig if approx._family == _lib.FAMILY_MF_GAUSSIAN else sig * sig * (approx.df / (approx.df - 2.0))
            corr[d:] = g_m * ubar + T - torch.diagonal(H) * scale2
        elif method == 'loo_diag_approx':
            corr[d:] = g_m * ubar
        grad = grad + corr
        if host:
            return float(value), grad.cpu().numpy()
        return value, grad

    def _engine(self, inject, S):
        """Cached fused step (engine.FusedStep, no optimiser) for this objective, or None when the
        (family, model) pair has none."""
        from .engine import FusedStep, fused_step_supported
        if not fused_step_supported(self):
            return None
        key = (bool(inject), int(S))
        eng = self._engines.get(key)
        if eng is not None and not eng.matches(self):
            eng = None
        if eng is None:
            try:
                eng = FusedStep(self, None, inject_base=inject, S=S)
            except NotImplementedError:
                return None
            self._engines[key] = eng
        return eng

    def _update_objective_and_grad(self):
        self._engines = {}
        if self.hessian_approx_method is not None:
            self._objective_and_grad = self._control_variate_objective
            return
        obj = _lib.OBJ_EXCLUSIVE_KL_PATH if self._use_path_deriv else _lib.OBJ_EXCLUSIVE_KL

        def objective_and_grad(var_param, base=None):
            host = is_host(var_param)
            S = self.num_mc_samples if base is None else int(base.shape[0] if hasattr(base, 'shape') else len(base))
            eng = self._engine(base is not None, S) if self.approx is not None and self.model is not None else None
            if eng is not None:
                # draw + reparameterise + pack | sweep | reduce + value + gradient: three kernels, one graph launch
                if base is not None:
                    eng.base.copy_(to_dev(base).reshape(S, -1))
                if host:
                    return eng.evaluate_host(var_param)
                eng.set_param(var_param)
                eng.run(1)
                return eng.value[0].clone(), eng.grad.clone()
            value, grad = _mf_objective(self.approx, self.model, self.num_mc_samples, obj, 0.0,
                                        var_param, base=base)
            if host:
                return _to_host(value, grad)
            return value, grad

        self._objective_and_grad = objective_and_grad

    def __call__(self, var_param, base=None):
        if self._objective_and_grad is None:
            raise RuntimeError("no objective and gradient available")
        if base is None:
            return self._objective_and_grad(var_param)
        return self._objective_and_grad(var_param, base=base)


class AlphaDivergence(StochasticVariationalObjective):
    """Log of the alpha-divergence (objectives.py:419-463)."""

    def __init__(self, approx, model, num_mc_samples, alpha):
        self._alpha = alpha
        super().__init__(approx, model, num_mc_samples)

    @property
    def alpha(self):
        return self._alpha

    def _update_objective_and_grad(self):
        def objective_grad_and_log_norm(var_param, base=None):
            host = is_host(var_param)
            # objectives.py:455: a fresh seed from the GLOBAL numpy RNG, shared by both passes
            seed = np.random.randint(2 ** 32, dtype=np.uint64) if base is None else None
            if seed is not None and getattr(self.model, 'sharded', False):
                # every rank must evaluate the SAME samples: rank 0's seed wins (ranks' global RNGs are not in step)
                seed = broadcast_seed(int(seed), getattr(self.model, 'process_group', None))
            value, grad = _mf_objective(self.approx, self.model, self.num_mc_samples, _lib.OBJ_ALPHA,
                                        self.alpha, var_param, base=base, seed=seed)
            if host:
                return _to_host(value, grad)
            return value, grad

        self._objective_and_grad = objective_grad_and_log_norm

    def __call__(self, var_param, base=None):
        if base is None:
            return self._objective_and_grad(var_param)
        return self._objective_and_grad(var_param, base=base)


class DISInclusiveKL(StochasticVariationalObjective):
    """Inclusive KL by distilled importance sampling (objectives.py:280-416).

    Forward-only in the model (no model gradient is ever needed): every `num_resampling_batches`-th
    call draws S samples, evaluates log q and log p, finds the tempering epsilon by bisection on the
    effective sample size, and then each call resamples from the tempered weights and differentiates
    -log q(lambda; x) at the FIXED samples (score terms).  Any family with a log density: the mean-field families,
    MultivariateT (both reparameterisations) and LRGaussian take the score from CUDA kernels (csrc/dis.cu,
    csrc/mvt_chol.cu, csrc/lr_score.cu), NVPFlow from torch autograd of its log density; NeuralNet has no density."""

    def __init__(self, approx, model, num_mc_samples, ess_target, temper_prior, temper_prior_params,
                 use_resampling=True, num_resampling_batches=1, w_clip_threshold=10):
        self._ess_target = ess_target
        self._w_clip_threshold = w_clip_threshold
        self._max_bisection_its = 50
        self._max_eps = self._eps = 1
        self._use_resampling = use_resampling
        self._num_resampling_batches = num_resampling_batches
        self._resampling_batch_size = max(1, self._ess_target // num_resampling_batches)
        self._objective_step = 0
        self._temper_prior = temper_prior
        self._temper_prior_params = temper_prior_params
        super().__init__(approx, model, num_mc_samples)

    # -- weights / ESS / bisection (objectives.py:317-366): one kernel launch on the S-vectors ----------------
    def _get_eps_and_weights(self, eps_guess, log_prior, log_p, log_q):
        S = int(log_q.numel())
        w = torch.empty(S, dtype=F64, device=log_q.device)
        out = torch.empty(4, dtype=F64, device=log_q.device)
        _lib.check(_lib.lib.vb_dis_bisection_f64(
            _lib.ptr(log_prior.contiguous()), _lib.ptr(log_p.contiguous()), _lib.ptr(log_q.contiguous()), S,
            float(eps_guess), float(self._max_eps), float(self._ess_target), int(self._max_bisection_its),
            _lib.ptr(w), _lib.ptr(out), _lib.stream()))
        eps, ess, zero, _ = out.cpu().numpy()
        if zero:
            raise ValueError('All weights zero! ' + 'Suggests overflow in importance density.')
        return float(eps), float(ess), w

    def _clip_weights(self, w):
        """Clip weights to `w_clip_threshold` x their sum, scaling the others up (objectives.py:368-386).
        The reference's branch for a threshold below 1 calls a float (`sum_unclipped(...)`, :385) and raises
        TypeError; this is the evident intent: clipped weights take the value that makes each of them exactly
        `threshold` x the new total."""
        thr = float(self._w_clip_threshold)
        w = w.clone()
        for _ in range(int(w.numel()) + 1):
            total = w.sum()
            if not bool((w > total * thr).any()):
                return w
            to_clip = w >= total * thr
            n_to_clip = int(to_clip.sum())
            sum_unclipped = w[~to_clip].sum()
            if float(sum_unclipped) == 0.0 or thr * n_to_clip >= 1.0:
                return w                        # impossible to clip further
            w[to_clip] = thr * sum_unclipped / (1.0 - thr * n_to_clip)
        return w

    def _resample_indices(self, S, p):
        """np.random.choice from the GLOBAL numpy RNG, as the reference (:408-409).  With a sharded model every
        rank must resample the same draws: rank 0 draws, the others receive."""
        try:
            idx = np.random.choice(S, size=self._resampling_batch_size, p=p)
        except ValueError:                     # probabilities off by more than numpy's tolerance: renormalise
            idx = np.random.choice(S, size=self._resampling_batch_size, p=p / p.sum())
        group = getattr(self.model, 'process_group', None)
        if getattr(self.model, 'sharded', False) and is_distributed(group):
            import torch.distributed as dist
            t = torch.as_tensor(idx, dtype=torch.int64, device=device())
            dist.broadcast(t, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
            idx = t.cpu().numpy()
        return idx

    def _score(self, vp, x, idx, w, scale):
        """(value, grad) = -sum_r c_r log q(x_r; lambda) and its gradient at the fixed samples, c_r = scale * w_r."""
        approx = self.approx
        d = approx.dim
        n = int(idx.numel()) if idx is not None else int(x.shape[0])
        if not isinstance(approx, _MeanField) and vp.numel() != approx.var_param_dim:
            raise ValueError('var_param has the wrong length')
        if isinstance(approx, NVPFlow):
            with torch.enable_grad():
                lam = vp.detach().clone().requires_grad_(True)
                lq = approx.log_density_t(lam, x if idx is None else x[idx])
                value = -scale * (lq if w is None else w * lq).sum()
                (grad,) = torch.autograd.grad(value, lam)
            return value.detach().reshape(1), grad
        out = torch.empty(1 + vp.numel(), dtype=F64, device=vp.device)
        lib, ptr = _lib.lib, _lib.ptr
        if isinstance(approx, MultivariateT):
            ws = torch.empty(lib.vb_mvt_score_workspace_bytes(n, d), dtype=torch.uint8, device=vp.device)
            _lib.check(lib.vb_mvt_score_f64(
                ptr(vp), ptr(x), ptr(idx), ptr(w), float(scale), n, d, float(approx.df), ptr(out[:1]), ptr(out[1:]),
                ptr(ws), ws.numel(), _lib.stream()))
        elif isinstance(approx, LRGaussian):
            from .convenience import _lr_projection
            P = _lr_projection(vp, approx)
            ws = torch.empty(lib.vb_lr_score_workspace_bytes(n, d, approx.k), dtype=torch.uint8, device=vp.device)
            _lib.check(lib.vb_lr_score_f64(
                ptr(vp), ptr(P), ptr(x), ptr(idx), ptr(w), float(scale), n, d, approx.k, ptr(out[:1]), ptr(out[1:]),
                ptr(ws), ws.numel(), _lib.stream()))
        else:
            ws = torch.empty(max(8, lib.vb_mf_score_workspace_bytes(d)), dtype=torch.uint8, device=vp.device)
            _lib.check(lib.vb_mf_score_f64(
                ptr(vp), ptr(x), ptr(idx), ptr(w), float(scale), n, d, approx._family,
                float(approx.df) if approx._family else 0.0, ptr(out[:1]), ptr(out[1:]), ptr(ws), ws.numel(),
                _lib.stream()))
        return out[:1], out[1:]

    def _mvt_draws(self, vp, S, base):
        """(x, log q(x)) for MultivariateT at a refresh: log q from the closed form at the draw,
        const - sum_i F_ii - (df + d)/2 log1p(|z/u|^2 / df), with no second eigensolver (sqrtm) and none at all
        (Cholesky).  In sqrtm mode an eigenvalue of Sigma at or below 1e-10, which the reference's log density drops
        from its pseudo-inverse, is refused, as streamed vi_diagnostics refuses it."""
        approx = self.approx
        d, df = approx.dim, float(approx.df)
        if vp.numel() != approx.var_param_dim:
            raise ValueError('var_param has the wrong length')
        chi2, z = approx.base_draws(S) if base is None else (to_dev(base[0]).reshape(-1), to_dev(base[1]))
        approx.last_base = (chi2, z)
        if approx.reparam == 'cholesky':
            x, _, zu2 = approx.chol_transform(vp, chi2, z)
        else:
            _, _, w, V = approx.decompose(vp)
            if float(w.min()) <= 1e-10:
                raise NotImplementedError('DISInclusiveKL for MultivariateT needs every eigenvalue of Sigma above 1e-10 '
                                          "in sqrtm mode; use reparam='cholesky'")
            x, _, zu2 = approx.transform(vp, chi2, z, w, V)
        i = torch.arange(d, device=vp.device)
        half_logdet = vp[d + i * (i + 3) // 2].sum()
        const = math.lgamma(0.5 * (df + d)) - math.lgamma(0.5 * df) - 0.5 * d * math.log(math.pi * df)
        return x, const - half_logdet - 0.5 * (df + d) * torch.log1p(zu2 / df)

    def _update_objective_and_grad(self):
        approx = self.approx
        if approx is not None and not isinstance(approx, (_MeanField, MultivariateT, LRGaussian, NVPFlow)):
            def unsupported(var_param, base=None):
                raise NotImplementedError('DISInclusiveKL needs a family with a log density')
            self._objective_and_grad = unsupported
            return

        def objective_and_grad(var_param, base=None):
            host = is_host(var_param)
            vp = to_dev(var_param)
            S = self.num_mc_samples
            if not self._use_resampling or self._objective_step % self._num_resampling_batches == 0:
                if isinstance(approx, MultivariateT):
                    x, self._state_log_q = self._mvt_draws(vp, S, base)
                else:
                    x = approx.sample(vp, S) if base is None else approx.sample(vp, S, base=base)
                    self._state_log_q = approx.log_density(vp, x)
                self._state_samples = x
                self._state_log_p = self.model(x)
                log_prior = self._temper_prior.log_density(to_dev(self._temper_prior_params), x)
                self._eps, ess, w = self._get_eps_and_weights(self._eps, log_prior, self._state_log_p,
                                                              self._state_log_q)
                w = self._clip_weights(w)               # a no-op for thresholds >= 1 (the default is 10)
                self._state_w = w
                self._state_w_sum = w.sum()
                self._state_w_normalized = w / self._state_w_sum
            self._objective_step += 1
            if not self._use_resampling:
                # -inner(w, log q) / S   (:405-406)
                value, grad = self._score(vp, self._state_samples, None, self._state_w, 1.0 / S)
            else:
                p = self._state_w_normalized.cpu().numpy()
                idx = self._resample_indices(S, p)
                idx_d = torch.as_tensor(idx, dtype=torch.int64, device=vp.device)
                # mean(-log q(x_idx)) * sum(w) / S   (:408-414)
                scale = float(self._state_w_sum) / S / idx_d.numel()
                value, grad = self._score(vp, self._state_samples, idx_d, None, scale)
            if host:
                return _to_host(value[0], grad)
            return value[0], grad

        self._objective_and_grad = objective_and_grad

    def __call__(self, var_param, base=None):
        if base is None:
            return self._objective_and_grad(var_param)
        return self._objective_and_grad(var_param, base=base)
