"""Fused ELBO-gradient step -- the three hot-path calls of the reference loop
(optimization.py:95-98: objective(var_param) -> descent_direction -> update) as ONE enqueue of
three kernels (ExclusiveKL) or five (AlphaDivergence: a forward-only sweep, the weights and a
weighted sweep) through `vb_mf_step_glm`, replayed from a CUDA graph.

Everything that changes from step to step lives on the device (draw-stream position or the
per-step seed, optimiser "first step" flag, history slot), so the host only replays graphs;
value / iterate / gradient histories are written by the step's last kernel into device rings.
With a sharded model the per-rank sums are exchanged inside the step's kernels through the
peer-memory communicator (parallel.Communicator) -- no NCCL call on the hot path.
"""
import ctypes
import gc
from ctypes import c_double, c_int32, c_int64, c_size_t, c_uint64, c_void_p

import numpy as np
import torch

from . import _lib
from ._tensor import F64, device, to_dev

__all__ = ['FusedStep', 'fused_step_supported']


class StepConfig(ctypes.Structure):
    _fields_ = [('family', c_int32), ('objective', c_int32), ('S', c_int32), ('d', c_int32),
                ('optimizer', c_int32), ('quantize', c_int32), ('inject_base', c_int32), ('reserved', c_int32),
                ('df', c_double), ('prior_sd', c_double), ('lr', c_double), ('beta1', c_double),
                ('beta2', c_double), ('jitter', c_double), ('seed', c_uint64), ('alpha', c_double)]


class StepBuffers(ctypes.Structure):
    _fields_ = [('var_param', c_void_p), ('opt_m', c_void_p), ('opt_nu', c_void_p), ('counters', c_void_p),
                ('base', c_void_p), ('theta', c_void_p), ('value', c_void_p), ('grad', c_void_p),
                ('logp', c_void_p), ('direction', c_void_p), ('value_hist', c_void_p), ('param_hist', c_void_p),
                ('grad_hist', c_void_p), ('dir_hist', c_void_p), ('hist_len', c_int64), ('ring', c_int64),
                ('seeds', c_void_p), ('seed_len', c_int64)]


class StepModel(ctypes.Structure):
    _fields_ = [('fast_handle', c_void_p), ('fast_workspace', c_void_p), ('fast_workspace_bytes', c_size_t),
                ('X', c_void_p), ('ldx', c_int64), ('y', c_void_p), ('N', c_int64), ('link', c_int32),
                ('reserved', c_int32), ('sweep_workspace', c_void_p), ('sweep_workspace_bytes', c_size_t)]



def _dp(t):
    return None if t is None else t.data_ptr()


def fused_step_supported(objective, optimizer=None):
    """True when `objective` (and `optimizer`) can run as the fused step: ExclusiveKL (entropy or
    path-derivative form, no control variates) or AlphaDivergence (finite, non-zero alpha) with a
    mean-field family on a GLM plugin, and plain RMSProp / Adam (or no optimiser)."""
    from .approximations import _MeanField
    from .models import GLMModel
    from .objectives import AlphaDivergence, ExclusiveKL
    from .optimization import Adam, RMSProp
    if type(objective) is ExclusiveKL:
        if objective.hessian_approx_method is not None:
            return False
    elif type(objective) is AlphaDivergence:
        try:
            alpha = float(objective.alpha)
        except (TypeError, ValueError):
            return False
        if not np.isfinite(alpha) or alpha == 0.0:
            return False
    else:
        return False
    if not isinstance(objective.approx, _MeanField) or not isinstance(objective.model, GLMModel):
        return False
    model = objective.model
    if model.path == 'fast' and objective.num_mc_samples > 256:
        return False
    if model.path != 'fast' and _lib.lib.vb_glm_sweep_workspace_bytes(model.N, model.dim, objective.num_mc_samples) == 0:
        return False
    if optimizer is not None and type(optimizer) not in (RMSProp, Adam):
        return False
    if optimizer is not None and getattr(optimizer, '_weight_decay', 0) not in (0, 0.0):
        pass        # weight decay only applies to 2-D parameters (optimization.py:99-100); ours are 1-D
    return True


class FusedStep(object):
    """Device-resident state of one (objective, optimiser) pair and its graph-replayed step.

    ring     : rows of the iterate / gradient / direction rings (0: none)
    hist_len : length of the value history (0: none)

    AlphaDivergence draws step t from a fresh Philox stream keyed by seeds[t % seed_len] (the
    reference draws a new global-numpy seed per call); set them with set_seeds() before the steps
    that use them.  ExclusiveKL draws from the family's own stream.
    """

    def __init__(self, objective, optimizer=None, ring=0, hist_len=0, want_logp=False, want_grad_hist=False,
                 want_dir_hist=False, inject_base=False, S=None):
        from .optimization import RMSProp
        if not fused_step_supported(objective, optimizer):
            raise NotImplementedError('this objective / optimiser pair has no fused step')
        self.objective, self.optimizer = objective, optimizer
        approx, model = objective.approx, objective.model
        self.approx, self.model = approx, model
        S, d = int(objective.num_mc_samples if S is None else S), int(approx.dim)
        if model.path == 'fast' and S > 256:
            raise NotImplementedError('the tensor-core sweep takes at most 256 samples')
        self.S, self.d, self.P = S, d, 2 * d
        dev = device()
        self.dev = dev
        self.inject = bool(inject_base)
        self.vp = torch.zeros(2 * d, dtype=F64, device=dev)
        self.counters = torch.zeros(4, dtype=torch.int64, device=dev)
        self.base = torch.zeros(S, d, dtype=F64, device=dev)
        self.theta = torch.zeros(S, d, dtype=F64, device=dev)
        self.out = torch.zeros(1 + 2 * d, dtype=F64, device=dev)        # [value | grad]: one D2H copy
        self.value, self.grad = self.out[:1], self.out[1:]
        self.logp = torch.zeros(S, dtype=F64, device=dev) if want_logp else None
        self.opt_kind = 0 if optimizer is None else (1 if type(optimizer) is RMSProp else 2)
        self.opt_nu = torch.zeros(2 * d, dtype=F64, device=dev) if self.opt_kind else None
        self.opt_m = torch.zeros(2 * d, dtype=F64, device=dev) if self.opt_kind == 2 else None
        self.ring, self.hist_len = int(ring), int(hist_len)
        self.value_hist = torch.zeros(max(1, self.hist_len), dtype=F64, device=dev) if hist_len else None
        self.param_hist = torch.zeros(self.ring, 2 * d, dtype=F64, device=dev) if ring else None
        self.grad_hist = torch.zeros(self.ring, 2 * d, dtype=F64, device=dev) if ring and want_grad_hist else None
        self.dir_hist = torch.zeros(self.ring, 2 * d, dtype=F64, device=dev) if ring and want_dir_hist else None
        self.direction = None
        # zero-initialised: the workspace carries the kernels' block ticket across calls
        self.ws = torch.zeros(_lib.lib.vb_mf_step_workspace_bytes(S, d), dtype=torch.uint8, device=dev)
        self.steps_done = 0
        self.path = model.path
        self.quantize = int(approx.quantize_draws)
        from .objectives import AlphaDivergence
        self.alpha = type(objective) is AlphaDivergence
        # pre, sweep, post; AlphaDivergence: pre, forward sweep, weights, weighted sweep, post
        self.launches_per_step = 5 if self.alpha else 3
        # AlphaDivergence: per-step seeds, one per history slot; the family's own stream is not used
        self.seed_len = max(1, self.hist_len) if self.alpha else 0
        self.seeds = torch.zeros(self.seed_len, dtype=torch.int64, device=dev) if self.alpha else None

        cfg = StepConfig()
        cfg.family = approx._family
        if self.alpha:
            cfg.objective = _lib.OBJ_ALPHA
            cfg.alpha = float(objective.alpha)
        else:
            cfg.objective = _lib.OBJ_EXCLUSIVE_KL_PATH if objective._use_path_deriv else _lib.OBJ_EXCLUSIVE_KL
        cfg.S, cfg.d = S, d
        cfg.optimizer = self.opt_kind
        cfg.quantize = self.quantize
        cfg.inject_base = int(self.inject)
        cfg.df = float(approx.df) if approx._family else 0.0
        cfg.prior_sd = float(model.prior_scale)
        if self.opt_kind == 1:
            cfg.lr, cfg.beta1, cfg.beta2, cfg.jitter = (float(optimizer._learning_rate), float(optimizer._beta), 0.0,
                                                        float(optimizer._jitter))
        elif self.opt_kind == 2:
            cfg.lr, cfg.beta1, cfg.beta2, cfg.jitter = (float(optimizer._learning_rate), float(optimizer._beta1),
                                                        float(optimizer._beta2), float(optimizer._jitter))
        cfg.seed = approx._seed
        self.cfg = cfg
        n = S * d
        self._stride = n + (n & 1)
        self._offset0 = 0
        self._rebase()

        mdl = StepModel()
        if model.path == 'fast':
            handle, _, fws = model._fast
            mdl.fast_handle = handle
            mdl.fast_workspace = fws.data_ptr()
            mdl.fast_workspace_bytes = fws.numel()
            self._keep = (fws,)
        else:
            need = _lib.lib.vb_glm_sweep_workspace_bytes(model.N, d, S)
            need = (need + 255) // 256 * 256
            sws = torch.empty(need + (S + 2 * d) * 8, dtype=torch.uint8, device=dev)
            mdl.X, mdl.ldx, mdl.y = model.X.data_ptr(), model.X.stride(0), model.y.data_ptr()
            mdl.N, mdl.link = model.N, model.link
            mdl.sweep_workspace, mdl.sweep_workspace_bytes = sws.data_ptr(), sws.numel()
            self._keep = (sws,)
            # pre, pack, sweep, 3 x reduce, post; AlphaDivergence: pre, forward (pack, sweep, reduce), weights,
            # weighted (pack, sweep, 3 x reduce), post
            self.launches_per_step = 11 if self.alpha else 7
        self.mdl = mdl

        self.comm = None
        if model.sharded:
            from .parallel import get_communicator, is_distributed
            if is_distributed(model.process_group):
                self.comm = get_communicator(model.process_group, (S + 2 * d) * 8)
                if self.comm is None:
                    raise NotImplementedError('no peer-memory communicator: the fused step cannot exchange its sums')
        b = StepBuffers()
        b.var_param, b.opt_m, b.opt_nu = _dp(self.vp), _dp(self.opt_m), _dp(self.opt_nu)
        b.counters = _dp(self.counters)
        b.base, b.theta, b.value, b.grad = _dp(self.base), _dp(self.theta), _dp(self.value), _dp(self.grad)
        b.logp, b.direction = _dp(self.logp), _dp(self.direction)
        b.value_hist, b.param_hist = _dp(self.value_hist), _dp(self.param_hist)
        b.grad_hist, b.dir_hist = _dp(self.grad_hist), _dp(self.dir_hist)
        b.hist_len, b.ring = self.hist_len, self.ring
        b.seeds, b.seed_len = _dp(self.seeds), self.seed_len
        self.buf = b
        self._graphs = {}
        self._warm = False           # a step has been enqueued eagerly: the lazy state a capture may not create exists
        self._pin_in = self._pin_out = None

    # -- state ---------------------------------------------------------------------------------
    def matches(self, objective):
        """Still valid for this objective's current model path / draw settings?"""
        return (self.model is objective.model and self.approx is objective.approx and self.path == objective.model.path
                and self.quantize == int(objective.approx.quantize_draws) and self.cfg.seed == objective.approx._seed
                and (self.path != 'fast' or self._keep[0] is objective.model._fast[2]))

    @property
    def _own_stream(self):
        """True when the steps draw from the family's own stream (ExclusiveKL without injected draws)."""
        return not self.inject and not self.alpha

    def set_seeds(self, t0, seeds):
        """Philox keys of steps t0 .. t0 + len(seeds) - 1 (AlphaDivergence), stored at t % seed_len.  A
        stream-ordered copy from pinned memory: it lands after the steps already enqueued and before the ones
        enqueued after it, and the host does not wait for it."""
        seeds = np.ascontiguousarray(seeds, dtype=np.uint64).reshape(-1)
        m = seeds.size
        if m == 0:
            return
        if m > self.seed_len:
            raise ValueError('more seeds than the engine keeps (%d)' % self.seed_len)
        # the pinned block is recycled by torch's host allocator only after the copy has run
        host = torch.from_numpy(seeds.view(np.int64)).pin_memory()
        a = int(t0) % self.seed_len
        n1 = min(m, self.seed_len - a)
        self.seeds[a:a + n1].copy_(host[:n1], non_blocking=True)
        if n1 < m:
            self.seeds[:m - n1].copy_(host[n1:], non_blocking=True)

    def draw_seeds(self, m):
        """Seeds of the next m AlphaDivergence steps from the global numpy RNG, as the reference draws one per call
        (objectives.py:455).  One vectorised draw of m seeds gives the values of m scalar draws and leaves the RNG
        in the same state.  On a sharded model rank 0's seeds are used everywhere (one broadcast for m steps)."""
        seeds = np.random.randint(2 ** 32, dtype=np.uint64, size=int(m))
        if getattr(self.model, 'sharded', False):
            from .parallel import broadcast_seeds
            seeds = broadcast_seeds(seeds, getattr(self.model, 'process_group', None))
        self.set_seeds(self.steps_done, seeds)

    def _rebase(self):
        """Point step `steps_done` of this engine at the family's current stream position."""
        self._offset0 = int(self.approx._offset) - self.steps_done * self._stride
        # stored modulo 2^64 (the kernel's unsigned arithmetic wraps the same way)
        v = self._offset0 % (1 << 64)
        self.counters[2] = v - (1 << 64) if v >= (1 << 63) else v

    def sync_stream_position(self):
        """Call before enqueuing when something else may have drawn from the family's stream."""
        if self._own_stream and int(self.approx._offset) != self._offset0 + self.steps_done * self._stride:
            self._rebase()

    def set_param(self, var_param):
        vp = to_dev(var_param).reshape(-1)
        if vp.numel() != self.P:
            raise ValueError('var_param has the wrong length')
        self.vp.copy_(vp)

    def set_learning_rate(self, lr):
        """A new learning rate invalidates the captured graphs (it is a kernel argument)."""
        if float(lr) != self.cfg.lr:
            self.cfg.lr = float(lr)
            self._graphs = {}

    def restart(self, keep_optimizer_state=False):
        """Restart the history index (and the optimiser's first-step flag); the draw stream keeps advancing."""
        pos = self._offset0 + self.steps_done * self._stride
        self.steps_done = 0
        self.counters[0] = 0
        if not keep_optimizer_state:
            self.counters[1] = 0
        if self._own_stream:
            self.approx._offset = pos
        self._rebase()

    def _after(self):
        if self._own_stream:
            self.approx._offset = self._offset0 + self.steps_done * self._stride
        self.approx.last_base = self.base

    # -- execution -----------------------------------------------------------------------------
    def enqueue(self):
        """One step on the current stream (no host synchronisation)."""
        _lib.check(_lib.lib.vb_mf_step_glm(ctypes.byref(self.cfg), ctypes.byref(self.buf), ctypes.byref(self.mdl),
                                           self.comm.handle if self.comm is not None else None,
                                           self.ws.data_ptr(), self.ws.numel(),
                                           torch.cuda.current_stream().cuda_stream))

    def _snapshot(self):
        return (self.vp.clone(), self.counters.clone(), None if self.opt_nu is None else self.opt_nu.clone(),
                None if self.opt_m is None else self.opt_m.clone())

    def _restore(self, snap):
        self.vp.copy_(snap[0])
        self.counters.copy_(snap[1])
        if snap[2] is not None:
            self.opt_nu.copy_(snap[2])
        if snap[3] is not None:
            self.opt_m.copy_(snap[3])

    def save_state(self):
        """Device copy of everything a step reads and advances (iterate, optimiser state, step and draw-stream
        counters), with the host's step count; no host synchronisation."""
        return self._snapshot(), self.steps_done

    def rewind(self, state):
        """Return to a state from save_state(): the steps that follow recompute what followed it, same draws included."""
        snap, self.steps_done = state
        self._restore(snap)
        self._after()

    def _capture(self, key, body):
        g = self._graphs.get(key)
        if g is None:
            if not self._warm:
                # one eager step outside the capture (lazy function attributes, tensor maps), device state rolled back
                snap = self._snapshot()
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    self.enqueue()
                torch.cuda.current_stream().wait_stream(side)
                torch.cuda.synchronize()
                self._restore(snap)
                torch.cuda.synchronize()
                self._warm = True
            g = torch.cuda.CUDAGraph()
            # Captured on a fresh side stream without synchronising the device: the capture only records launches,
            # so the host builds the graph while the steps already enqueued keep the GPU busy.
            # No garbage collection inside the capture: a collected object that owns device resources (an old
            # graph, a model handle) would call cudaFree / cudaGraphExecDestroy, which a capture forbids.
            gc_was_on = gc.isenabled()
            gc.disable()
            try:
                with torch.cuda.stream(torch.cuda.Stream()):
                    g.capture_begin(capture_error_mode='thread_local')
                    try:
                        body()
                    finally:
                        g.capture_end()
            finally:
                if gc_was_on:
                    gc.enable()
            self._graphs[key] = g
        return g

    def run(self, n, unroll=8, use_graph=True):
        """n steps: graphs of `unroll` steps plus single-step graphs for the remainder."""
        n = int(n)
        self.sync_stream_position()
        if not use_graph:
            for _ in range(n):
                self.enqueue()
            self._warm = self._warm or n > 0
        else:
            m = n
            big = m // unroll if unroll > 1 else 0
            if not self._warm and ((big and unroll not in self._graphs) or (m - big * unroll and 1 not in self._graphs)):
                # the first step runs eagerly and counts: it creates what a capture may not (module loads, function
                # attributes, tensor maps), so no rolled-back warm-up step is spent (eager and replayed steps are
                # bitwise equal)
                self.enqueue()
                self._warm = True
                m -= 1
                big = m // unroll if unroll > 1 else 0
            if big:
                g = self._capture(unroll, lambda: [self.enqueue() for _ in range(unroll)])
                for _ in range(big):
                    g.replay()
            rest = m - big * unroll
            if rest:
                g = self._capture(1, self.enqueue)
                for _ in range(rest):
                    g.replay()
        self.steps_done += n
        self._after()

    def evaluate_host(self, var_param):
        """objective(var_param) for a numpy var_param: ONE graph launch carrying the H2D copy of the
        parameter (pinned), the step's three kernels and the D2H copy of [value | grad] (pinned)."""
        if self._pin_in is None:
            self._pin_in = torch.empty(self.P, dtype=F64).pin_memory()
            self._pin_out = torch.empty(1 + self.P, dtype=F64).pin_memory()
        vp = np.asarray(var_param, dtype=np.float64).reshape(-1)
        if vp.size != self.P:
            raise ValueError('var_param has the wrong length')
        self.sync_stream_position()

        def body():
            self.vp.copy_(self._pin_in, non_blocking=True)
            self.enqueue()
            self._pin_out.copy_(self.out, non_blocking=True)

        g = self._capture('host', body)
        self._pin_in.numpy()[:] = vp
        g.replay()
        torch.cuda.current_stream().synchronize()
        self.steps_done += 1
        self._after()
        h = self._pin_out.numpy()
        return float(h[0]), h[1:].copy()

    def check_comm(self):
        if self.comm is not None and _lib.lib.vb_comm_error(self.comm.handle):
            raise RuntimeError('viabel_b200: a peer never arrived at the in-kernel all-reduce')

    # -- history access (device tensors, oldest first) -----------------------------------------
    def last_rows(self, hist, count):
        """The `count` most recent rows of a ring, oldest first."""
        count = int(min(count, self.steps_done, self.ring))
        end = self.steps_done % self.ring
        if count <= end:
            return hist[end - count:end]
        return torch.cat([hist[self.ring - (count - end):], hist[:end]])
