"""Stochastic optimisers -- mirror of viabel/optimization.py's SGD family (:52-476).

`optimize()` keeps the variational parameter, the optimiser state and all histories on the
device; RMSProp and Adam use the fused CUDA step (state update + parameter update in one
launch).  `descent_direction(grad)` is kept for drop-in use with numpy arrays or tensors and
reproduces the reference's first-step behaviour (SURVEY.md App. C).
"""
from abc import ABC, abstractmethod
from collections import defaultdict

import numpy as np
import torch
import tqdm

from . import _lib
from ._tensor import F64, device, to_dev

__all__ = ['Optimizer', 'StochasticGradientOptimizer', 'RMSProp', 'Adam', 'Adagrad', 'WindowedAdagrad',
           'AveragedRMSProp', 'AveragedAdam']


def _sqrt(x):
    return torch.sqrt(x) if isinstance(x, torch.Tensor) else np.sqrt(x)


def _to_numpy_results(results):
    out = {}
    for key, hist in results.items():
        if isinstance(hist, list) and len(hist) and isinstance(hist[0], torch.Tensor):
            out[key] = torch.stack(list(hist)).cpu().numpy()       # keeps the parameter's own shape
        elif isinstance(hist, torch.Tensor):
            out[key] = hist.cpu().numpy()
        else:
            out[key] = np.array(hist)
    return out


class Optimizer(ABC):
    @abstractmethod
    def optimize(self, n_iters, objective, init_param, **kwargs):
        """Return a dict with at least `opt_param`."""


class StochasticGradientOptimizer(Optimizer):
    """Plain SGD and the base of the adaptive methods (optimization.py:52-144)."""

    def __init__(self, learning_rate, *, weight_decay=0, iterate_avg_prop=0.2, diagnostics=False):
        self._learning_rate = learning_rate
        self._weight_decay = weight_decay
        if iterate_avg_prop is not None and (iterate_avg_prop > 1.0 or iterate_avg_prop <= 0.0):
            raise ValueError('"iterate_avg_prop" must be None or between 0 and 1')
        self._iterate_avg_prop = iterate_avg_prop
        self._diagnostics = diagnostics
        self.progress = True
        self.reset_state()

    def reset_state(self):
        pass

    def descent_direction(self, grad):
        return grad

    def _fused_step(self, var_param, grad, want_dir):
        """In-place `var_param -= lr * direction` on device tensors; returns direction or None.
        Subclasses with a CUDA step override this."""
        direction = self.descent_direction(grad)
        var_param -= self._learning_rate * direction
        return direction if want_dir else None

    # -- fused path: the whole loop as graph replays of the three-kernel step (engine.FusedStep) -------
    def _export_state(self, eng):
        """Optimiser state -> engine (the state persists across optimize() calls, as in the reference)."""

    def _import_state(self, eng):
        """Engine -> optimiser state."""

    def _history_length(self, n_iters):
        """Length of the reference's trimmed iterate list after n_iters iterations (optimization.py:103-106)."""
        iap = self._iterate_avg_prop
        if iap is None:
            return n_iters if self._diagnostics else 0
        L = 0
        for k in range(n_iters):
            L += 1
            if L > iap * k:
                L -= 1
        return L

    def _optimize_fused(self, n_iters, objective, init_param):
        from .engine import FusedStep
        iap = self._iterate_avg_prop
        L = self._history_length(n_iters)
        window = max(1, int((n_iters - 1) * iap)) if iap is not None else 0
        ring = n_iters if self._diagnostics else max(L, window, 1)
        eng = FusedStep(objective, self, ring=ring, hist_len=n_iters, want_dir_hist=self._diagnostics)
        eng.set_param(init_param)
        self._export_state(eng)
        done = 0
        chunk = 100 if self.progress else 1000
        bar = tqdm.tqdm(total=n_iters, disable=not self.progress)
        try:
            while done < n_iters:
                m = min(chunk, n_iters - done)
                if eng.alpha:
                    eng.draw_seeds(m)
                eng.run(m)
                done += m
                if self.progress:
                    bar.update(m)
                    recent = eng.value_hist[max(0, done - 1000):done]
                    bar.set_description('average loss = {:,.5g}'.format(float(recent.mean())))
        except (KeyboardInterrupt, StopIteration):  # pragma: no cover
            pass
        finally:
            bar.close()
        torch.cuda.current_stream().synchronize()
        eng.check_comm()
        self._import_state(eng)
        results = {'value_history': eng.value_hist[:done].cpu().numpy()}
        k = done - 1
        if (self._diagnostics or iap is not None) and done > 0:
            keep = self._history_length(done)
            results['variational_param_history'] = eng.last_rows(eng.param_hist, keep).cpu().numpy()
        if self._diagnostics:
            results['descent_dir_history'] = eng.last_rows(eng.dir_hist, done).cpu().numpy()
        if iap is not None and done > 0 and self._history_length(done) > 0:
            w = min(max(1, int(k * iap)), self._history_length(done))
            results['opt_param'] = eng.last_rows(eng.param_hist, w).mean(dim=0).cpu().numpy()
        else:
            results['opt_param'] = eng.vp.cpu().numpy()
        return results

    def optimize(self, n_iters, objective, init_param, init_hamflow_model_param=None,
                 init_hamflow_rho_param=None):
        """The reference loop (optimization.py:83-127) with device-resident state."""
        from .engine import fused_step_supported
        from .objectives import VariationalObjective
        if n_iters > 0 and np.ndim(init_param) == 1 and fused_step_supported(objective, self):
            rng = np.random.get_state()
            try:
                return self._optimize_fused(n_iters, objective, init_param)
            except NotImplementedError:
                np.random.set_state(rng)         # AlphaDivergence seeds drawn for the fused step: draw them again
        var_param = to_dev(init_param).clone()
        iap = self._iterate_avg_prop
        results = defaultdict(list)
        plain_update = type(objective).update is VariationalObjective.update \
            if isinstance(objective, VariationalObjective) else False
        k = -1
        bar = tqdm.trange(n_iters, disable=not self.progress)
        try:
            for k in bar:
                value, grad = objective(var_param)
                if not isinstance(grad, torch.Tensor):      # host objective (user code)
                    grad = to_dev(grad)
                    value = torch.as_tensor(float(value), dtype=F64, device=grad.device)
                if plain_update:
                    direction = self._fused_step(var_param, grad, self._diagnostics)
                else:
                    direction = self.descent_direction(grad)
                    var_param = to_dev(objective.update(var_param, self._learning_rate * direction))
                if var_param.dim() == 2:
                    var_param *= (1 - self._weight_decay)
                results['value_history'].append(value.detach().reshape(()))
                if self._diagnostics or iap is not None:
                    results['variational_param_history'].append(var_param.clone())
                    if iap is not None and len(results['variational_param_history']) > iap * k:
                        results['variational_param_history'].pop(0)
                if self._diagnostics:
                    results['descent_dir_history'].append(direction.clone())
                if self.progress and k % 10 == 0:
                    recent = torch.stack(results['value_history'][max(0, k - 1000):k + 1])
                    bar.set_description('average loss = {:,.5g}'.format(float(recent.mean())))
        except (KeyboardInterrupt, StopIteration):  # pragma: no cover
            pass
        finally:
            bar.close()
        if iap is not None and len(results['variational_param_history']):
            window = max(1, int(k * iap))
            tail = torch.stack(results['variational_param_history'][-window:])
            results['opt_param'] = tail.mean(dim=0)
        else:
            # (for n_iters <= 5 the reference's window is empty and it returns NaN; the last
            # iterate is returned instead)
            results['opt_param'] = var_param.clone()
        return _to_numpy_results(results)


class RMSProp(StochasticGradientOptimizer):
    """RMSProp (optimization.py:147-197): nu starts at grad**2."""

    def __init__(self, learning_rate, *, weight_decay=0, iterate_avg_prop=0.2, beta=0.9, jitter=1e-8,
                 diagnostics=False):
        self._beta = beta
        self._jitter = jitter
        super().__init__(learning_rate, weight_decay=weight_decay, iterate_avg_prop=iterate_avg_prop,
                         diagnostics=diagnostics)

    def reset_state(self):
        self._avg_grad_sq = None

    def descent_direction(self, grad):
        g2 = grad ** 2
        nu = g2 if self._avg_grad_sq is None else self._avg_grad_sq
        nu = nu * self._beta
        nu = nu + (1. - self._beta) * g2
        self._avg_grad_sq = nu
        return grad / _sqrt(self._jitter + nu)

    def _export_state(self, eng):
        if self._avg_grad_sq is not None:
            eng.opt_nu.copy_(to_dev(self._avg_grad_sq))
            eng.counters[1] = 1
        else:
            eng.counters[1] = 0

    def _import_state(self, eng):
        if eng.steps_done > 0:
            self._avg_grad_sq = eng.opt_nu.clone()

    def _fused_step(self, var_param, grad, want_dir):
        first = self._avg_grad_sq is None or not isinstance(self._avg_grad_sq, torch.Tensor)
        if first:
            self._avg_grad_sq = torch.empty_like(grad)
        direction = torch.empty_like(grad) if want_dir else None
        _lib.check(_lib.lib.vb_rmsprop_step_f64(
            _lib.ptr(var_param), _lib.ptr(grad), _lib.ptr(self._avg_grad_sq), _lib.ptr(direction),
            grad.numel(), float(self._learning_rate), float(self._beta), float(self._jitter), int(first),
            _lib.stream()))
        return direction


class Adam(StochasticGradientOptimizer):
    """Adam (optimization.py:260-326), including the first-step aliasing of `momentum = grad`."""

    def __init__(self, learning_rate, *, beta1=0.9, beta2=0.999, jitter=1e-8, iterate_avg_prop=0.2,
                 diagnostics=False):
        self._beta1 = beta1
        self._beta2 = beta2
        self._jitter = jitter
        super().__init__(learning_rate, iterate_avg_prop=iterate_avg_prop, diagnostics=diagnostics)

    def reset_state(self):
        self._momentum = None
        self._avg_grad_sq = None

    def descent_direction(self, grad):
        b1, b2 = self._beta1, self._beta2
        if self._momentum is None:
            scaled = grad * b1                       # the aliased array after `momentum *= beta1`
            m = scaled + (1. - b1) * scaled
            nu = (grad ** 2) * b2
            nu = nu + (1. - b2) * m ** 2
        else:
            m = self._momentum * b1
            m = m + (1. - b1) * grad
            nu = self._avg_grad_sq * b2
            nu = nu + (1. - b2) * grad ** 2
        self._momentum, self._avg_grad_sq = m, nu
        return m / _sqrt(self._jitter + nu)

    def _export_state(self, eng):
        if self._momentum is not None:
            eng.opt_m.copy_(to_dev(self._momentum))
            eng.opt_nu.copy_(to_dev(self._avg_grad_sq))
            eng.counters[1] = 1
        else:
            eng.counters[1] = 0

    def _import_state(self, eng):
        if eng.steps_done > 0:
            self._momentum = eng.opt_m.clone()
            self._avg_grad_sq = eng.opt_nu.clone()

    def _fused_step(self, var_param, grad, want_dir):
        first = self._momentum is None or not isinstance(self._momentum, torch.Tensor)
        if first:
            self._momentum = torch.empty_like(grad)
            self._avg_grad_sq = torch.empty_like(grad)
        direction = torch.empty_like(grad) if want_dir else None
        _lib.check(_lib.lib.vb_adam_step_f64(
            _lib.ptr(var_param), _lib.ptr(grad), _lib.ptr(self._momentum), _lib.ptr(self._avg_grad_sq),
            _lib.ptr(direction), grad.numel(), float(self._learning_rate), float(self._beta1),
            float(self._beta2), float(self._jitter), int(first), _lib.stream()))
        return direction


class AveragedRMSProp(StochasticGradientOptimizer):
    """optimization.py:200-258 (beta_k = 1 - 1/k)."""

    def __init__(self, learning_rate, *, jitter=1e-8, diagnostics=False, component_wise=True):
        self._jitter = jitter
        self._component_wise = component_wise
        super().__init__(learning_rate, diagnostics=diagnostics)

    def reset_state(self):
        self._avg_grad_sq = None
        self._t = None

    def descent_direction(self, grad):
        g2 = grad ** 2
        if self._avg_grad_sq is None:
            nu, t = g2, 1
        else:
            nu, t = self._avg_grad_sq, self._t + 1
        beta = 1 - 1 / t
        nu = nu * beta + (1. - beta) * g2
        self._avg_grad_sq, self._t = nu, t
        denom = nu if self._component_wise else nu.sum()
        return grad / _sqrt(self._jitter + denom)


class AveragedAdam(StochasticGradientOptimizer):
    """optimization.py:328-396."""

    def __init__(self, learning_rate, *, beta1=0.9, jitter=1e-8, diagnostics=False, component_wise=True):
        self._beta1 = beta1
        self._jitter = jitter
        self._component_wise = component_wise
        super().__init__(learning_rate, diagnostics=diagnostics)

    def reset_state(self):
        self._momentum = None
        self._avg_grad_sq = None
        self._t = None

    def descent_direction(self, grad):
        b1 = self._beta1
        if self._momentum is None:
            # same aliasing as Adam: grad is scaled in place before it is reused
            scaled = grad * b1
            m = scaled + (1. - b1) * scaled
            g_eff2 = m ** 2
            nu, t = grad ** 2, 1
        else:
            m = self._momentum * b1 + (1. - b1) * grad
            g_eff2 = grad ** 2
            nu, t = self._avg_grad_sq, self._t + 1
        beta2 = 1 - 1 / t
        nu = nu * beta2 + (1. - beta2) * g_eff2
        self._momentum, self._avg_grad_sq, self._t = m, nu, t
        denom = nu if self._component_wise else nu.sum()
        return m / _sqrt(self._jitter + denom)


class Adagrad(StochasticGradientOptimizer):
    """optimization.py:398-433."""

    def __init__(self, learning_rate, *, weight_decay=0, jitter=1e-8, iterate_avg_prop=0.2, diagnostics=False):
        self._jitter = jitter
        super().__init__(learning_rate, weight_decay=weight_decay, iterate_avg_prop=iterate_avg_prop,
                         diagnostics=diagnostics)

    def reset_state(self):
        self._sum_grad_sq = 0

    def descent_direction(self, grad):
        self._sum_grad_sq = self._sum_grad_sq + grad ** 2
        return grad / _sqrt(self._jitter + self._sum_grad_sq)


class WindowedAdagrad(StochasticGradientOptimizer):
    """optimization.py:435-476."""

    def __init__(self, learning_rate, *, weight_decay=0, window_size=10, jitter=1e-8, diagnostics=False):
        self._window_size = window_size
        self._jitter = jitter
        super().__init__(learning_rate, weight_decay=weight_decay, diagnostics=diagnostics)

    def reset_state(self):
        self._history = []

    def descent_direction(self, grad):
        self._history.append(grad ** 2)
        if len(self._history) > self._window_size:
            self._history.pop(0)
        mean_sq = sum(self._history) / len(self._history)
        return grad / _sqrt(self._jitter + mean_sq)


# ---------------------------------------------------------------------------------------------
# FASO / RAABBVI: host control loops (optimization.py:479-931).  Per iteration they make exactly
# the three hot-path calls objective(vp) -> descent_direction -> update; the iterate history
# stays on the device and only the windows inspected by the convergence checks are copied back.
# ---------------------------------------------------------------------------------------------
import time as _time

from ._mc_diagnostics import MCSE, R_hat_convergence_check

__all__ += ['FASO', 'RAABBVI']


def _window(hist, W):
    """Last W iterates as a host [W, P] array."""
    return torch.stack(hist[-int(W):]).cpu().numpy()


class FASO(Optimizer):
    """Fixed-learning-rate stochastic optimisation with R-hat / MCSE stopping (:479-633)."""

    #: device memory the iterate ring of the general (unfused) loop may take; 0 forces the reference's host lists
    _device_ring_bytes = 48e9

    def __init__(self, sgo, *, mcse_threshold=0.1, W_min=200, ESS_min=None, k_check=None):
        if not isinstance(sgo, StochasticGradientOptimizer):
            raise ValueError('sgo must be a subclass of StochasticGradientOptimizer')
        self._sgo = sgo
        self._mcse_threshold = mcse_threshold
        self._W_min = W_min
        self._ESS_min = W_min // 8 if ESS_min is None else ESS_min
        self._k_check = W_min if k_check is None else k_check
        if mcse_threshold <= 0:
            raise ValueError('"mcse_threshold" must be greater than zero')
        if W_min <= 0:
            raise ValueError('"W_min" must be greater than zero')
        if self._k_check <= 0:
            raise ValueError('"k_check" must be greater than zero')
        if self._ESS_min <= 0:
            raise ValueError('"ESS_min" must be greater than zero')

    def _mcse_of_window(self, iterates, objective, dim_param):
        from .approximations import MFGaussian
        W = iterates.shape[0]
        if isinstance(objective.approx, MFGaussian):
            # MCSE(mu / sigma, log sigma), constant coordinates dropped (:575-590)
            dim = int(dim_param / 2)
            still = (iterates[W - 2, :] - iterates[W - 1, :]) == 0
            if np.any(still):
                iterates = np.delete(iterates, np.argwhere(still), 1)
            mean_log_sd = np.mean(iterates[:, -dim:], axis=0)
            ess, mcse = MCSE(iterates)
            mcse = np.concatenate((mcse[:dim] / np.exp(mean_log_sd), mcse[-dim:]))
            return ess, mcse
        return MCSE(iterates)

    # -- fused path: graph-replayed steps between the checks, statistics on the device ring -------------
    def _optimize_fused(self, n_iters, objective, init_param):
        from ._mc_diagnostics import RingStats
        from .approximations import MFGaussian
        from .engine import FusedStep
        sgo = self._sgo
        diagnostics = sgo._diagnostics
        host_init = np.array(init_param.detach().cpu().numpy() if isinstance(init_param, torch.Tensor)
                             else init_param, dtype=np.float64)
        P = host_init.size
        eng = FusedStep(objective, sgo, ring=n_iters, hist_len=n_iters, want_grad_hist=True, want_dir_hist=diagnostics)
        eng.set_param(host_init)
        sgo._export_state(eng)
        stats = RingStats(eng.param_hist, n_iters, P)
        k_conv = k_stopped = k_Rhat = None
        W_check = None
        mcse = ess = None
        hist = defaultdict(list)
        iterate_average = host_init.copy()
        if diagnostics:
            hist['iterate_average_k_history'].append(0)
            hist['iterate_average_history'].append(iterate_average)
        opt_time = 0.0
        progress = getattr(sgo, 'progress', True)
        bar = tqdm.tqdm(total=n_iters, disable=not progress)
        done = 0                               # iterations completed; the reference's k is done - 1
        try:
            while done < n_iters:
                # run up to and including the next iteration at which the reference looks at the history
                k_next = (done + self._k_check - 1) // self._k_check * self._k_check        # next multiple >= done
                if k_conv is not None:
                    k_next = min(k_next, max(k_conv + W_check, done))
                k_next = min(k_next, n_iters - 1)
                t0 = _time.perf_counter()
                if eng.alpha:
                    eng.draw_seeds(k_next + 1 - done)
                eng.run(k_next + 1 - done)
                torch.cuda.current_stream().synchronize()
                opt_time += _time.perf_counter() - t0
                bar.update(k_next + 1 - done)
                done = k_next + 1
                k = k_next
                if k_conv is None and k % self._k_check == 0:
                    W_upper = int(0.95 * k)
                    if W_upper > self._W_min:
                        windows = np.linspace(self._W_min, W_upper, num=5, dtype=int)
                        ok, best_W = stats.convergence_check(done, windows)
                        iterate_average = stats.window_mean(done, best_W).cpu().numpy()
                        if diagnostics:
                            hist['iterate_average_k_history'].append(k)
                            hist['iterate_average_history'].append(iterate_average)
                        if ok:
                            k_Rhat, k_conv, W_check = k, k - best_W, best_W
                if k_conv is not None and k - k_conv == W_check:
                    W = W_check
                    t1 = _time.perf_counter()
                    ess, mcse, mean = stats.mcse(done, W)
                    iterate_average = mean
                    if isinstance(objective.approx, MFGaussian):
                        # MCSE(mu / sigma, log sigma), constant coordinates dropped (optimization.py:575-590); the
                        # statistics are per column, so the reference's np.delete acts on the per-column vectors
                        dim = int(P / 2)
                        last2 = eng.last_rows(eng.param_hist, 2)
                        still = (last2[0] == last2[1]).cpu().numpy()
                        if np.any(still):
                            drop = np.argwhere(still)
                            ess, mcse, mean_kept = np.delete(ess, drop), np.delete(mcse, drop), np.delete(mean, drop)
                        else:
                            mean_kept = mean
                        mcse = np.concatenate((mcse[:dim] / np.exp(mean_kept[-dim:]), mcse[-dim:]))
                    mcse_time = _time.perf_counter() - t1
                    if diagnostics:
                        if k not in hist['iterate_average_k_history']:
                            hist['iterate_average_k_history'].append(k)
                            hist['iterate_average_history'].append(iterate_average)
                        hist['ess_and_mcse_k_history'].append(k)
                        hist['ess_history'].append(ess)
                        hist['mcse_history'].append(mcse)
                    if np.max(mcse) < self._mcse_threshold and np.min(ess) > self._ESS_min:
                        k_stopped = k
                        break
                    ratio = (opt_time / max(k, 1)) / (mcse_time / W)
                    W_check = int(max(1.05, 1 + 1 / np.sqrt(1 + ratio)) * W_check + 1)
                if progress and k % self._k_check == 0:
                    recent = eng.value_hist[max(0, k - 1000):k + 1]
                    bar.set_description('average loss = {:,.5g} | R hat {}|'.format(
                        float(recent.mean()), 'converged' if k_conv is not None else 'not converged'))
        except (KeyboardInterrupt, StopIteration):  # pragma: no cover
            pass
        finally:
            bar.close()
        torch.cuda.current_stream().synchronize()
        eng.check_comm()
        sgo._import_state(eng)
        self._report(k_stopped, k_conv, mcse, ess)
        results = {'value_history': eng.value_hist[:done].cpu().numpy(),
                   'grad_history': eng.last_rows(eng.grad_hist, done).cpu().numpy(),
                   'variational_param_history': eng.last_rows(eng.param_hist, done).cpu().numpy()}
        if diagnostics:
            results['descent_dir_history'] = eng.last_rows(eng.dir_hist, done).cpu().numpy()
        for key, v in hist.items():
            results[key] = np.array(v)
        results['k_conv'] = k_conv
        results['k_Rhat'] = k_Rhat
        results['k_stopped'] = k_stopped
        results['opt_param'] = np.asarray(iterate_average)
        return results

    @staticmethod
    def _report(k_stopped, k_conv, mcse, ess):
        if k_stopped is None:
            if k_conv is None:
                print('WARNING: stationarity not reached after maximum number of iterations')
                print('WARNING: try incresing the learning rate or the maximum number of iterations')
            else:
                print('WARNING: stationarity reached but MCSE too large and/or ESS too small')
                if mcse is not None:
                    print('WARNING: maximum MCSE = {:.3g}'.format(np.max(mcse)))
                    print('WARNING: minimum ESS = {:.1f}'.format(np.min(ess)))
        else:
            print('Convergence reached at iteration', k_stopped)

    def optimize(self, n_iters, objective, init_param):
        from .engine import fused_step_supported
        from .objectives import VariationalObjective
        sgo = self._sgo
        if (n_iters > 0 and np.ndim(init_param) == 1 and fused_step_supported(objective, sgo)
                and 3 * n_iters * np.size(init_param) * 8 < 8e9):
            rng = np.random.get_state()
            try:
                return self._optimize_fused(n_iters, objective, init_param)
            except NotImplementedError:
                np.random.set_state(rng)         # AlphaDivergence seeds drawn for the fused step: draw them again
        diagnostics = sgo._diagnostics
        k_conv = k_stopped = k_Rhat = None
        lr = sgo._learning_rate
        host_init = np.array(init_param.detach().cpu().numpy() if isinstance(init_param, torch.Tensor)
                             else init_param, dtype=np.float64)
        vp = to_dev(host_init).clone()
        plain_update = isinstance(objective, VariationalObjective) and \
            type(objective).update is VariationalObjective.update
        hist = defaultdict(list)
        iterate_average = host_init.copy()
        if diagnostics:
            hist['iterate_average_k_history'].append(0)
            hist['iterate_average_history'].append(iterate_average)
        opt_time = 0.0
        mcse = ess = None
        W_check = None
        # Iterate history: a device ring [n_iters, P] with the batched device statistics (csrc/faso.cu) whenever it
        # fits -- the reference's host lists + per-parameter MCSE loop (optimization.py:546, _mc_diagnostics.py:119)
        # cannot work at BASELINE configs[3]'s 2.1 M parameters; host lists remain the fallback for huge n_iters * P
        from ._mc_diagnostics import RingStats
        from .approximations import MFGaussian
        P = host_init.size
        ring = stats = None
        if n_iters > 0 and n_iters * P * 8 <= self._device_ring_bytes:
            ring = torch.empty(n_iters, P, dtype=F64, device=vp.device)
            stats = RingStats(ring, n_iters, P)
        progress = getattr(sgo, 'progress', True)
        bar = tqdm.trange(n_iters, disable=not progress)
        done = 0
        try:
            for k in bar:
                t0 = _time.perf_counter()
                value, grad = objective(vp)
                if not isinstance(grad, torch.Tensor):
                    grad = to_dev(grad)
                    value = torch.as_tensor(float(value), dtype=F64, device=grad.device)
                hist['value_history'].append(value.detach().reshape(()))
                hist['grad_history'].append(grad)
                if plain_update:
                    direction = sgo._fused_step(vp, grad, diagnostics)
                else:
                    direction = sgo.descent_direction(grad)
                    vp = to_dev(objective.update(vp, lr * direction))
                if ring is not None:
                    ring[k].copy_(vp.reshape(-1))
                else:
                    hist['variational_param_history'].append(vp.clone())
                done = k + 1
                if diagnostics:
                    hist['descent_dir_history'].append(direction.clone())
                opt_time += _time.perf_counter() - t0

                if k_conv is None and k % self._k_check == 0:
                    W_upper = int(0.95 * k)
                    if W_upper > self._W_min:
                        windows = np.linspace(self._W_min, W_upper, num=5, dtype=int)
                        if stats is not None:
                            ok, best_W = stats.convergence_check(done, windows)
                            iterate_average = stats.window_mean(done, best_W).cpu().numpy()
                        else:
                            recent = _window(hist['variational_param_history'], W_upper)
                            ok, best_W = R_hat_convergence_check(recent, windows)
                            iterate_average = np.mean(recent[-best_W:], axis=0)
                        if diagnostics:
                            hist['iterate_average_k_history'].append(k)
                            hist['iterate_average_history'].append(iterate_average)
                        if ok:
                            k_Rhat, k_conv, W_check = k, k - best_W, best_W

                if k_conv is not None and k - k_conv == W_check:
                    W = W_check
                    if stats is not None:
                        t1 = _time.perf_counter()
                        ess, mcse, iterate_average = stats.mcse(done, W)
                        if isinstance(objective.approx, MFGaussian):
                            # MCSE(mu / sigma, log sigma), constant coordinates dropped (optimization.py:575-590)
                            dim = int(P / 2)
                            still = (ring[k - 1] == ring[k]).cpu().numpy()
                            mean_kept = iterate_average
                            if np.any(still):
                                drop = np.argwhere(still)
                                ess, mcse, mean_kept = np.delete(ess, drop), np.delete(mcse, drop), np.delete(mean_kept, drop)
                            mcse = np.concatenate((mcse[:dim] / np.exp(mean_kept[-dim:]), mcse[-dim:]))
                        mcse_time = _time.perf_counter() - t1
                    else:
                        iterates = _window(hist['variational_param_history'], W)
                        iterate_average = np.mean(iterates, axis=0)
                        t1 = _time.perf_counter()
                        ess, mcse = self._mcse_of_window(iterates, objective, host_init.size)
                        mcse_time = _time.perf_counter() - t1
                    if diagnostics and k not in hist['iterate_average_k_history']:
                        hist['iterate_average_k_history'].append(k)
                        hist['iterate_average_history'].append(iterate_average)
                    if diagnostics:
                        hist['ess_and_mcse_k_history'].append(k)
                        hist['ess_history'].append(ess)
                        hist['mcse_history'].append(mcse)
                    if np.max(mcse) < self._mcse_threshold and np.min(ess) > self._ESS_min:
                        k_stopped = k
                        break
                    ratio = (opt_time / k) / (mcse_time / W)
                    W_check = int(max(1.05, 1 + 1 / np.sqrt(1 + ratio)) * W_check + 1)
                if progress and k % self._k_check == 0:
                    recent = torch.stack(hist['value_history'][max(0, k - 1000):k + 1])
                    bar.set_description('average loss = {:,.5g} | R hat {}|'.format(
                        float(recent.mean()), 'converged' if k_conv is not None else 'not converged'))
        except (KeyboardInterrupt, StopIteration):  # pragma: no cover
            pass
        finally:
            bar.close()
        self._report(k_stopped, k_conv, mcse, ess)
        results = _to_numpy_results(hist)
        if ring is not None:
            results['variational_param_history'] = ring[:done].cpu().numpy()
        results['k_conv'] = k_conv
        results['k_Rhat'] = k_Rhat
        results['k_stopped'] = k_stopped
        results['opt_param'] = iterate_average
        return results


def _posterior_mean_regression(y, x, w, rho, fixed_kappa=None):
    """Deterministic replacement for RAABBVI's Stan/NUTS fit of
        y_n ~ N(log_c + 2 log(rho^-kappa - 1) + 2 kappa x_n, sigma) ^ w_n,
        kappa ~ U(0,1), log_c ~ Cauchy(0,10), sigma ~ half-Cauchy(0,10)
    (stan_models/weighted_lin_regression*.stan, optimization.py:677-725): posterior means of
    kappa and log_c by quadrature on a (kappa, log_c, sigma) grid."""
    y, x, w = (np.asarray(v, dtype=np.float64) for v in (y, x, w))
    kap = np.array([fixed_kappa]) if fixed_kappa is not None else (np.arange(200) + 0.5) / 200
    off = 2 * np.log(rho ** (-kap) - 1)[:, None] + 2 * kap[:, None] * x[None, :]     # [K, N]
    resid0 = y[None, :] - off                                                          # = log_c + noise
    centre = np.sum(w * resid0, axis=1) / np.sum(w)
    spread = max(np.sqrt(np.max(np.sum(w * (resid0 - centre[:, None]) ** 2, axis=1) / np.sum(w))), 1e-3)
    lc = np.linspace(centre.min() - 12 * spread - 1, centre.max() + 12 * spread + 1, 400)
    sig = np.exp(np.linspace(np.log(spread * 1e-2), np.log(spread * 1e2 + 10), 160))
    # sum_n w_n (r_n - lc)^2 = A - 2 lc B + lc^2 C
    A = np.sum(w * resid0 ** 2, axis=1)[:, None]
    B = np.sum(w * resid0, axis=1)[:, None]
    C = np.sum(w)
    sse = A - 2 * lc[None, :] * B + lc[None, :] ** 2 * C                               # [K, L]
    logpost = (-0.5 * sse[:, :, None] / sig[None, None, :] ** 2 - C * np.log(sig)[None, None, :]
               - np.log1p((lc[None, :, None] / 10) ** 2) - np.log1p((sig[None, None, :] / 10) ** 2)
               + np.log(sig)[None, None, :])            # + log sigma: grid is uniform in log sigma
    p = np.exp(logpost - logpost.max())
    p /= p.sum()
    kappa = float(np.sum(p.sum(axis=(1, 2)) * kap))
    log_c = float(np.sum(p.sum(axis=(0, 2)) * lc))
    return kappa, np.exp(log_c)


class RAABBVI(FASO):
    """Robust, automated, accurate BBVI: FASO runs at a decreasing learning rate with the
    inefficiency-index termination rule (optimization.py:635-931).  The NUTS regression for
    (kappa, c) is replaced by deterministic quadrature over the same posterior."""

    def __init__(self, sgo, *, rho=0.5, iters0=1000, accuracy_threshold=0.1, inefficiency_threshold=1.0,
                 init_rmsprop=False, **kwargs):
        super().__init__(sgo, **kwargs)
        self._iters0 = iters0
        self._rho = rho
        self._accuracy_threshold = accuracy_threshold
        self._inefficiency_threshold = inefficiency_threshold
        self._init_rmsprop = init_rmsprop
        if rho < 0 or rho > 1:
            raise ValueError('"rho" must be between zero and one')

    def _averaged(self):
        return isinstance(self._sgo, (AveragedRMSProp, AveragedAdam))

    def weighted_linear_regression(self, model, y, x, s=9, a=0.25, n_chains=4):
        N = len(y)
        w = np.array(1 / (1 + np.arange(N)[::-1] ** 2 / s) ** a)
        kappa, c = _posterior_mean_regression(y, x, w, self._rho, 1.0 if self._averaged() else None)
        return None, kappa, c

    def wls(self, x, y, s=9, a=0.25):
        n = y.size
        Xd = np.column_stack((np.ones(n), x))
        w = 1 / (1 + np.arange(n)[::-1] ** 2 / s ** 2) ** a
        # least squares on the sqrt(w)-scaled system; with a single point (which the reference
        # hands to np.linalg.inv of a singular 2x2, :754) this is the minimum-norm fit
        sw = np.sqrt(w)
        beta = np.linalg.lstsq(sw[:, None] * Xd, sw * np.asarray(y, dtype=float), rcond=None)[0]
        return beta[0], beta[1]

    def convg_iteration_trend_detection(self, slope):
        return bool(slope < 0)

    def optimize(self, K_max, objective, init_param):
        if not objective.approx.supports_kl:
            print('WARNING: approximation family does not support KL. Using FASO.', flush=True)
            return super().optimize(K_max, objective, init_param)
        sgo = self._sgo
        diagnostics = sgo._diagnostics
        rho = self._rho
        k_new, k, k_total, k_add = -1, 0, 0, 0
        k_stopped_final = None
        current = np.array(init_param, dtype=np.float64, copy=True)
        h = defaultdict(list)
        h['iterate_average_curr_hist'].append(current)
        h['k_mcse'].append(0)
        stopped = False
        index = None
        try:
            while not stopped:
                K_max -= (k_new + 1)
                previous = current
                if k == 0 and self._init_rmsprop:
                    first = RMSProp(learning_rate=sgo._learning_rate, diagnostics=diagnostics)
                    first.progress = getattr(sgo, 'progress', True)
                    opt = FASO(sgo=first).optimize(K_max, objective, current)
                else:
                    opt = FASO.optimize(self, K_max, objective, current)
                if opt['k_stopped'] is not None and k != 0:
                    h['conv_iters_hist'].append(opt['k_stopped'])
                current = opt['opt_param']
                h['iterate_average_curr_hist'].append(current)
                k_new = opt['k_stopped']
                shift = k_new is not None
                h['k_Rhat'].append(opt['k_Rhat'] + k_add if opt['k_Rhat'] is not None and shift else opt['k_Rhat'])
                h['k_conv'].append(opt['k_conv'] + k_add if opt['k_conv'] is not None and shift else opt['k_conv'])
                h['k_mcse'].append(k_new + k_add if shift else k_new)
                for key in ('variational_param_history', 'value_history', 'grad_history'):
                    h[key].extend(opt[key])
                if diagnostics:
                    h['descent_dir_history'].extend(opt['descent_dir_history'])
                    if opt['k_conv'] is not None:
                        h['ess_history'].extend(opt.get('ess_history', []))
                        h['mcse_history'].extend(opt.get('mcse_history', []))
                        h['final_mcse_history'].append(h['mcse_history'][-1] if len(h['mcse_history'])
                                                       else h['mcse_history'])
                    if k == 0:
                        h['iterate_average_k_history'].extend(opt['iterate_average_k_history'])
                        h['iterate_average_history'].extend(opt['iterate_average_history'])
                    else:
                        h['iterate_average_k_history'].extend(opt['iterate_average_k_history'][1:] + k_add)
                        h['iterate_average_history'].extend(opt['iterate_average_history'][1:, :])
                k_add = h['iterate_average_k_history'][-1] if len(h['iterate_average_k_history']) else k_add
                if k_new is None:
                    break
                k_total += k_new
                sgo._learning_rate *= rho
                self._mcse_threshold *= rho
                if self._averaged():
                    sgo.reset_state()
                if len(h['learning_rate_hist']) > 0:
                    approx = objective.approx
                    h['SKL_history'].append(approx.kl(previous, current) + approx.kl(current, previous))
                    y_wlr = np.log(h['SKL_history'])
                    x_wlr = np.log(h['learning_rate_hist'])
                    _, kappa, c = self.weighted_linear_regression(None, y_wlr, x_wlr)
                    h['kappa_hist'].append(kappa)
                    h['c_hist'].append(c)
                    if len(h['learning_rate_hist']) > 1:
                        last_lr = h['learning_rate_hist'][-1]
                        relative_skl = rho ** kappa + self._accuracy_threshold / (np.sqrt(c) * last_lr ** kappa)
                        curr_iters = h['conv_iters_hist'][-1]
                        _, slope = self.wls(np.log(h['learning_rate_hist']), np.log(h['conv_iters_hist']))
                        if self.convg_iteration_trend_detection(slope):
                            xs, ys = h['learning_rate_hist'], h['conv_iters_hist']
                        else:
                            xs, ys = h['learning_rate_hist'][1:], h['conv_iters_hist'][1:]
                        b0, b1 = self.wls(np.log(xs), np.log(ys))
                        pred_iters = int(np.exp(b0) * (rho * last_lr) ** b1)
                        h['predicted_iters_hist'].append(pred_iters)
                        relative_iters = pred_iters / (curr_iters + self._iters0)
                        index = relative_skl * relative_iters
                        h['stopping_crt'].append(index)
                        if index > self._inefficiency_threshold:
                            stopped = True
                            k_stopped_final = k_total
                            h['k_stopped_final_hist'].append(k_total)
                            break
                h['learning_rate_hist'].append(sgo._learning_rate)
                k += 1
        except (KeyboardInterrupt, StopIteration):  # pragma: no cover
            pass
        if stopped:
            print('Termination rule reached at iteration', k_total)
            print('Inefficiency Index:', index)
        else:
            print('WARNING: maximum number of iterations reached before stopping rule was triggered')
        results = {key: np.array(v) for key, v in h.items() if key not in ('k_Rhat', 'k_mcse', 'k_conv')}
        results['opt_param'] = current
        results['k_stopped_final'] = k_stopped_final
        results['k_Rhat'] = h['k_Rhat']
        results['k_mcse'] = h['k_mcse']
        results['k_conv'] = h['k_conv']
        return results
