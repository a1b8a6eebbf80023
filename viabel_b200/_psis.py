"""Pareto smoothed importance sampling -- drop-in mirror of viabel/_psis.py (psislw :113-209).

The n log-weights stay on the device; the reference's full argsort is replaced by a
threshold + radix-select pipeline (see csrc/psis.cu).  gpdfitnew / gpinv / sumlogs keep their
reference signatures as thin host helpers for small arrays.
"""
from ctypes import c_void_p

import numpy as np
import torch

from . import _lib
from ._tensor import F64, device, is_host, to_dev

__all__ = ['psislw', 'psislw_device', 'psislw_batch_device', 'psis_batch_max_n', 'psislw_sharded', 'PsisShard',
           'psisloo', 'gpdfitnew', 'gpinv', 'sumlogs']

R_KHAT, R_SIGMA, R_N2, R_CUTOFF, R_LSE, R_MAX, R_STATUS, R_SUMV, R_SUMEXP2V, R_M, R_NCAND, R_SMOOTHED = range(12)

_ws_cache = {}


def _workspace(n, reff):
    key = (int(n), float(reff), torch.cuda.current_device())
    ws = _ws_cache.get(key)
    if ws is None:
        nbytes = _lib.lib.vb_psis_workspace_bytes(n, reff)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=device())
        if len(_ws_cache) > 8:
            _ws_cache.clear()
        _ws_cache[key] = ws
    return ws


def psislw_device(lw, out=None, Reff=1.0, want_tail=False, exact=False):
    """PSIS of one column of log-weights held in a contiguous CUDA float64 tensor.

    Enqueues the whole pipeline without a host sync.  Returns (out, result, tail_idx, tail_rank)
    where result is the 16-slot device vector described in include/viabel_b200.h.  `out` may be
    `lw` itself (in place) or None (k-hat only)."""
    n = lw.numel()
    if n <= 1:
        raise ValueError("More than one log-weight needed.")
    result = torch.empty(16, dtype=F64, device=lw.device)
    tail_idx = tail_rank = None
    if want_tail:
        cap = _lib.lib.vb_psis_tail_capacity(n, Reff)
        tail_idx = torch.empty(cap, dtype=torch.int64, device=lw.device)
        tail_rank = torch.empty(cap, dtype=torch.int32, device=lw.device)
    ws = _workspace(n, Reff)
    _lib.check(_lib.lib.vb_psislw_f64(_lib.ptr(lw), _lib.ptr(out), n, float(Reff), int(exact),
                                      _lib.ptr(result), _lib.ptr(tail_idx), _lib.ptr(tail_rank),
                                      _lib.ptr(ws), ws.numel(), _lib.stream()))
    return out, result, tail_idx, tail_rank


def psis_batch_max_n(Reff=1.0):
    """Longest column the batched kernel holds in one CTA's shared memory (falls with Reff: M can reach 0.2 n)."""
    return int(_lib.lib.vb_psis_batch_max_n(float(Reff)))


def _column_major(t):
    """Leading dimension of a 2-D tensor whose columns are contiguous, else None."""
    n, m = t.shape
    if m <= 1:
        return n if (n <= 1 or t.stride(0) == 1) else None
    return t.stride(1) if (t.stride(0) == 1 and t.stride(1) >= n) else None


def psislw_batch_device(lw2d, out=None, Reff=1.0, want_loo=False, want_result=False):
    """PSIS of every column of an n x m CUDA float64 matrix in one launch (vb_psislw_batch_f64).

    lw2d and out must have contiguous columns (stride(0) == 1, any leading dimension >= n), as a transposed
    contiguous [m, n] tensor or a Fortran-ordered copy has.  `out` may be lw2d itself or None (no output written).
    Enqueues one kernel without a host sync and returns device tensors (out, khat[m], result[m, 16] or None,
    loo[m] or None); loo[j] is log-sum-exp_i(out[i, j] - lw2d[i, j]), psisloo's term for lw2d = -log_lik.
    n must not exceed psis_batch_max_n(Reff) (NotImplementedError)."""
    if lw2d.dim() != 2 or lw2d.dtype != F64 or not lw2d.is_cuda:
        raise ValueError('psislw_batch_device needs a 2-D CUDA float64 tensor')
    n, m = lw2d.shape
    ld = _column_major(lw2d)
    if ld is None:
        raise ValueError('psislw_batch_device needs contiguous columns (stride(0) == 1)')
    ldo = n
    if out is not None:
        if tuple(out.shape) != (n, m) or out.dtype != F64 or out.device != lw2d.device:
            raise ValueError('out must be an n x m float64 tensor on the device of lw2d')
        ldo = _column_major(out)
        if ldo is None:
            raise ValueError('out needs contiguous columns (stride(0) == 1)')
    khat = torch.empty(m, dtype=F64, device=lw2d.device)
    result = torch.empty((m, 16), dtype=F64, device=lw2d.device) if want_result else None
    loo = torch.empty(m, dtype=F64, device=lw2d.device) if want_loo else None
    if m == 0:
        return out, khat, result, loo
    _lib.check(_lib.lib.vb_psislw_batch_f64(
        c_void_p(lw2d.data_ptr()), max(ld, n), n, m, float(Reff),
        None if out is None else c_void_p(out.data_ptr()), max(ldo, n),
        _lib.ptr(khat), _lib.ptr(result), _lib.ptr(loo), _lib.stream()))
    return out, khat, result, loo


def _psis_columns(cols, Reff):
    """Columns longer than the batched kernel holds: the one-column pipeline on every row of the contiguous [m, n]
    tensor `cols` (smoothed in place), all enqueued before ONE read of the [m, 16] result rows; the columns whose
    sampled threshold missed (status 1, nothing written) are rerun in exact mode.  Returns k-hat (numpy)."""
    m, n = cols.shape
    res = torch.empty((m, 16), dtype=F64, device=cols.device)
    ws = _workspace(n, Reff)

    def run(i, exact):
        _lib.check(_lib.lib.vb_psislw_f64(_lib.ptr(cols[i]), _lib.ptr(cols[i]), n, float(Reff), int(exact),
                                          _lib.ptr(res[i]), None, None, _lib.ptr(ws), ws.numel(), _lib.stream()))
    for i in range(m):
        run(i, False)
    r = res.cpu().numpy()
    redo = np.flatnonzero(r[:, R_STATUS] == 1)
    for i in redo:
        run(i, True)
    if redo.size:
        r[redo] = res[torch.as_tensor(redo, device=cols.device)].cpu().numpy()
    bad = np.flatnonzero(r[:, R_STATUS] != 0)
    if bad.size:
        raise RuntimeError('viabel_b200: PSIS failed with status %d' % int(r[bad[0], R_STATUS]))
    return r[:, R_KHAT].copy()


def _psis_column(col, out, Reff, want_tail):
    o, result, ti, tr = psislw_device(col, out, Reff, want_tail)
    res = result.cpu().numpy()
    if res[R_STATUS] == 1:          # sampled threshold missed the tail: exact radix passes
        o, result, ti, tr = psislw_device(col, out, Reff, want_tail, exact=True)
        res = result.cpu().numpy()
    if res[R_STATUS] != 0:
        raise RuntimeError('viabel_b200: PSIS failed with status %d' % int(res[R_STATUS]))
    return res, ti, tr


def psislw(lw, Reff=1.0, overwrite_lw=False, return_tail=False):
    """Pareto smoothed importance sampling (_psis.py:113-209).

    lw: array of n log weights, or n x m for m sets (numpy array or CUDA tensor).
    Returns (lw_out, kss) like the reference: smoothed, normalised log weights and the Pareto
    tail index/indices.  With overwrite_lw=True a CUDA tensor (or F-contiguous numpy array) is
    smoothed in place.  return_tail=True (1-D only) appends (tail_idx, tail_rank)."""
    host = is_host(lw)
    if host:
        lw_np = np.asarray(lw)
        ndim = lw_np.ndim
    else:
        ndim = lw.dim()
    if ndim not in (1, 2):
        raise ValueError("Argument `lw` must be 1 or 2 dimensional.")
    n = lw_np.shape[0] if host else lw.shape[0]
    if n <= 1:
        raise ValueError("More than one log-weight needed.")

    if ndim == 1:
        col = to_dev(lw_np) if host else lw.to(F64).contiguous()
        inplace = (not host) and overwrite_lw and col.data_ptr() == lw.data_ptr()
        out = col if (inplace or host) else torch.empty_like(col)
        res, ti, tr = _psis_column(col, out, Reff, return_tail)
        k = float(res[R_KHAT])
        if host:
            out_np = out.cpu().numpy()
            if overwrite_lw and isinstance(lw, np.ndarray) and lw.flags.f_contiguous and lw.dtype == np.float64:
                lw[...] = out_np
                out_np = lw
            ret = (out_np, k)
        else:
            ret = (out, k)
        if return_tail:
            n2 = int(res[R_N2])
            ret = ret + (ti[:n2].cpu().numpy() if host else ti[:n2], tr[:n2].cpu().numpy() if host else tr[:n2])
        return ret

    if return_tail:
        raise ValueError('return_tail is only available for 1-D input')
    m = lw_np.shape[1] if host else lw.shape[1]
    # columns that fit one CTA's shared memory: one launch for the whole matrix; longer ones: the one-column pipeline
    batched = n <= psis_batch_max_n(Reff)
    if host:
        inplace = overwrite_lw and isinstance(lw, np.ndarray) and lw_np.flags.f_contiguous and lw_np.dtype == np.float64
        cols = torch.from_numpy(np.ascontiguousarray(lw_np.T, dtype=np.float64)).to(device())     # [m, n]
        if batched:
            _, khat, _, _ = psislw_batch_device(cols.t(), cols.t(), Reff)
            kss = khat.cpu().numpy()
        else:
            kss = _psis_columns(cols, Reff)
        res = cols.cpu().numpy().T                   # F-contiguous n x m
        if inplace:
            lw_np[...] = res
            return lw_np, kss
        return res, kss
    src = lw.to(F64)
    if batched and _column_major(src) is not None:
        # columns already contiguous (an F-ordered or transposed tensor, any leading dimension): no staging copy
        if overwrite_lw and src.data_ptr() == lw.data_ptr():
            out = src
        else:
            out = torch.empty((m, n), dtype=F64, device=src.device).t()
        _, khat, _, _ = psislw_batch_device(src, out, Reff)
        kss = khat.cpu().numpy()
    else:
        cols = src.t().contiguous()                  # [m, n]: each set contiguous
        if cols.data_ptr() == lw.data_ptr() and not overwrite_lw:
            cols = cols.clone()                      # [n,1] and F-ordered inputs: t() is already contiguous -> a view
        if batched:
            _, khat, _, _ = psislw_batch_device(cols.t(), cols.t(), Reff)
            kss = khat.cpu().numpy()
        else:
            kss = _psis_columns(cols, Reff)
        out = cols.t()
    if overwrite_lw and out.data_ptr() != lw.data_ptr():
        lw.copy_(out)
        out = lw
    return out, kss


class PsisShard:
    """One rank's part of a draw-sharded PSIS (SURVEY.md 8(e)): `lw` holds the n_local consecutive
    draws starting at global index `idx_off` out of n_global.  The three stages mirror
    vb_psis_dist_local / _global / _apply; the exchange between the first two (an all-gather of
    the fixed-size records) is the caller's -- see `psislw_sharded`.  Kept as an object so that a
    test can drive several shards inside one process."""

    def __init__(self, lw, idx_off, n_global, Reff=1.0, world=1, rank=0):
        if lw.dim() != 1 or lw.dtype != F64 or not lw.is_cuda or not lw.is_contiguous():
            raise ValueError('PsisShard needs a contiguous 1-D CUDA float64 tensor')
        if lw.numel() <= 1:
            raise ValueError("More than one log-weight needed.")
        self.lw, self.idx_off, self.n_global = lw, int(idx_off), int(n_global)
        self.reff, self.world, self.rank = float(Reff), int(world), int(rank)
        nbytes = _lib.lib.vb_psis_dist_workspace_bytes(lw.numel(), self.n_global, self.reff, self.world)
        self.reclen = _lib.lib.vb_psis_dist_record_doubles(self.n_global, self.reff)
        if nbytes == 0 or self.reclen == 0:
            raise ValueError('invalid shard sizes')
        self.ws = torch.empty(nbytes, dtype=torch.uint8, device=lw.device)
        self.record = torch.empty(self.reclen, dtype=F64, device=lw.device)
        self.result = torch.empty(16, dtype=F64, device=lw.device)

    def local(self, exact=False):
        """Stage 1 -> this rank's record (device tensor of `reclen` doubles)."""
        _lib.check(_lib.lib.vb_psis_dist_local(
            _lib.ptr(self.lw), self.lw.numel(), self.idx_off, self.n_global, self.reff, self.world, int(exact),
            _lib.ptr(self.record), _lib.ptr(self.ws), self.ws.numel(), _lib.stream()))
        return self.record

    def global_(self, records):
        """Stage 2 on the records of all ranks ([world * reclen] doubles, rank order)."""
        if records.numel() != self.world * self.reclen or records.dtype != F64 or not records.is_contiguous():
            raise ValueError('records must be world x reclen contiguous float64')
        _lib.check(_lib.lib.vb_psis_dist_global(
            _lib.ptr(records), self.lw.numel(), self.n_global, self.reff, self.world, _lib.ptr(self.result),
            _lib.ptr(self.ws), self.ws.numel(), _lib.stream()))
        return self.result

    def apply(self, out):
        """Stage 3: writes this rank's smoothed, normalised log-weights (out may be None or lw);
        result slots 7 and 8 hold this rank's share of the moments."""
        _lib.check(_lib.lib.vb_psis_dist_apply(
            _lib.ptr(self.lw), _lib.ptr(out), self.lw.numel(), self.idx_off, self.n_global, self.reff, self.world,
            self.rank, _lib.ptr(self.result), _lib.ptr(self.ws), self.ws.numel(), _lib.stream()))
        return self.result


def psislw_sharded(lw_local, Reff=1.0, out=None, group=None, want_out=True, sizes=None):
    """PSIS of ONE column of log-weights whose draws are sharded over the ranks of `group`
    (rank r holds consecutive draws; sizes may differ).  Same result as `psislw` on the
    concatenation (_psis.py:113-209): every rank runs pass A and a local cutoff on its draws, the
    ranks all-gather their top-(M+1) records (16 (M+1) bytes each), the global cutoff / GPD fit /
    log-sum-exp run replicated, and pass B writes each rank's part.  `sizes` (per-rank draw
    counts) saves the one host round trip that discovers them.

    Returns (out_local, khat, result) with result the 16-slot host vector of include/viabel_b200.h,
    its moments (slots 7, 8) summed over ranks."""
    import torch.distributed as dist
    from . import parallel
    rank, ws = parallel.world(group)
    lw_local = lw_local.to(F64).contiguous()
    if sizes is None:
        sz = torch.zeros(ws, dtype=torch.int64, device=lw_local.device)
        sz[rank] = lw_local.numel()
        sizes = parallel.allreduce_sum_(sz, group).cpu().tolist()
    if len(sizes) != ws or sizes[rank] != lw_local.numel():
        raise ValueError('sizes does not match the process group / local shard')
    shard = PsisShard(lw_local, sum(sizes[:rank]), sum(sizes), Reff, ws, rank)
    if out is None and want_out:
        out = torch.empty_like(lw_local)
    for exact in (False, True):
        rec = shard.local(exact)
        if ws > 1:
            recs = torch.empty(ws * shard.reclen, dtype=F64, device=rec.device)
            dist.all_gather_into_tensor(recs, rec, group=group)
        else:
            recs = rec
        shard.global_(recs)
        result = shard.apply(out)
        parallel.allreduce_sum_(result[R_SUMV:R_SUMEXP2V + 1], group)
        res = result.cpu().numpy()               # the only host sync; status is identical on every rank
        if res[R_STATUS] == 0:
            return out, float(res[R_KHAT]), res
        if res[R_STATUS] != 1:
            break
    raise RuntimeError('viabel_b200: PSIS failed with status %d' % int(res[R_STATUS]))


def gpinv(p, k, sigma):
    """Inverse generalised Pareto distribution function (_psis.py:335-377)."""
    p = np.asarray(p, dtype=np.float64)
    x = np.full(p.shape, np.nan)
    if sigma <= 0:
        return x
    ok = (p > 0) & (p < 1)
    if abs(k) < np.finfo(float).eps:
        x[ok] = -np.log1p(-p[ok])
    else:
        x[ok] = np.expm1(-k * np.log1p(-p[ok])) / k
    x *= sigma
    x[p == 0] = 0
    x[p == 1] = np.inf if k >= 0 else -sigma / k
    return x


def gpdfitnew(x, sort=True, sort_in_place=False, return_quadrature=False):
    """Zhang-Stephens estimate of the generalised Pareto parameters (_psis.py:212-332); host
    helper for small arrays -- psislw runs the same fit on the device."""
    x = np.asarray(x, dtype=np.float64)
    if x.ndim != 1 or len(x) <= 1:
        raise ValueError("Invalid input array.")
    if sort is True:
        if sort_in_place:
            x.sort()
            xs = x
        else:
            xs = np.sort(x)
    elif sort is False:
        xs = x
    else:
        xs = x[sort]
    n = len(xs)
    m = 30 + int(np.sqrt(n))
    j = np.arange(1, m + 1, dtype=float) - 0.5
    bs = (1 - np.sqrt(m / j)) / (3 * xs[int(n / 4 + 0.5) - 1]) + 1 / xs[-1]
    ks = np.mean(np.log1p(-bs[:, None] * xs), axis=1)
    with np.errstate(all='ignore'):
        L = n * (np.log(-bs / ks) - ks - 1)
        w = 1 / np.sum(np.exp(L - L[:, None]), axis=1)
    keep = w >= 10 * np.finfo(float).eps
    w, bsk = w[keep], bs[keep]
    w = w / w.sum()
    b = np.sum(bsk * w)
    k = np.mean(np.log1p(-b * xs))
    sigma = -k / b
    k = k * n / (n + 10) + 5 / (n + 10)
    if return_quadrature:
        kq = np.mean(np.log1p(-bsk[:, None] * xs), axis=1) * n / (n + 10) + 5 / (n + 10)
        return k, sigma, kq, w
    return k, sigma


def psisloo(log_lik, **kwargs):
    """PSIS leave-one-out log predictive densities (_psis.py:69-110): log_lik is n x m (n posterior draws of the m
    log-likelihood terms); every column is one PSIS problem on the raw log-weights -log_lik.  Returns (loo, loos[m],
    ks[m]): Python float and numpy arrays for numpy input, device tensors (loo 0-d) for a CUDA tensor.  log_lik is
    never modified.  Further keyword arguments go to psislw (Reff).

    When n <= psis_batch_max_n(Reff) the whole matrix is one launch of the batched kernel without an output array:
    one read of log_lik, and loos come out of the kernel (sumlogs(lw_smoothed + log_lik) per column)."""
    host = is_host(log_lik)
    ll = np.asarray(log_lik, dtype=np.float64) if host else log_lik
    if ll.ndim != 2:
        raise ValueError('log_lik must be an n x m array')
    n, m = ll.shape
    Reff = kwargs.get('Reff', 1.0)
    if n > 1 and n <= psis_batch_max_n(Reff):
        if host:
            cols = torch.from_numpy(np.ascontiguousarray(ll.T)).to(device())       # [m, n]
            cols.neg_()
        else:
            cols = torch.empty((m, n), dtype=F64, device=ll.device)
            torch.neg(ll.to(F64).t(), out=cols)
        _, khat, _, loos = psislw_batch_device(cols.t(), None, Reff, want_loo=True)
        loo = loos.sum()
        if host:
            return float(loo), loos.cpu().numpy(), khat.cpu().numpy()
        return loo, loos, khat
    kwargs['overwrite_lw'] = True
    if host:
        lw, ks = psislw(np.asfortranarray(-ll), **kwargs)
        loos = sumlogs(lw + ll, axis=0)
        return loos.sum(), loos, ks
    # columns longer than the batched kernel holds: the one-column pipeline smooths them, sumlogs of the m columns
    # (one reduction each) runs as device tensor operations
    lw, ks = psislw(-ll.to(F64), **kwargs)
    t = lw + ll.to(F64)
    mx = t.max(dim=0, keepdim=True).values
    loos = torch.log(torch.exp(t - mx).sum(dim=0)) + mx[0]
    return loos.sum(), loos, torch.as_tensor(ks, device=ll.device)


def sumlogs(x, axis=None, out=None):
    """log(sum(exp(x))) (_psis.py:380-396)."""
    x = np.asarray(x)
    mx = x.max(axis=axis, keepdims=True)
    r = np.log(np.sum(np.exp(x - mx), axis=axis)) + np.squeeze(mx)
    if out is not None:
        out[...] = r
        return out
    return r
