"""Multi-GPU plumbing for the sharded hot path (SURVEY.md 8(e)): one process per GPU,
torch.distributed over NCCL (gloo in the CPU tests of this host logic).

* ELBO gradient: observations are sharded by rows; every rank draws identical base variates
  (same Philox seed / offset), so the only exchange is a sum of the per-rank sweep outputs
  [ll(S), gmu(d), ge(d)] -- a <= 10 KB, latency-bound all-reduce.
* PSIS: draws are sharded; ranks exchange their candidate lists (all-gather) and a handful of
  scalars; the smoothed weights stay sharded.
"""
import ctypes
import warnings

import numpy as np
import torch
import torch.distributed as dist

__all__ = ['is_distributed', 'world', 'shard_rows', 'allreduce_sum_', 'allgather_ragged', 'Communicator',
           'get_communicator', 'broadcast_seed']


def is_distributed(group=None):
    return dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1


def world(group=None):
    """(rank, world_size); (0, 1) when torch.distributed is not initialised."""
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(group), dist.get_world_size(group)
    return 0, 1


def shard_rows(n, rank, world_size):
    """Contiguous, balanced [lo, hi) slice of n rows for `rank` (sizes differ by at most one)."""
    if not 0 <= rank < world_size:
        raise ValueError('rank out of range')
    base, rem = divmod(int(n), int(world_size))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


class Communicator(object):
    """Peer-memory communicator of libviabel_b200 (`vb_comm_*`, include/viabel_b200.h): every rank's
    exchange buffer is mapped into every other rank through CUDA IPC; collectives are single kernels
    that store into the peers' buffers over NVLink.  torch.distributed only carries the 64-byte
    handles once, at construction (a collective call: every rank of `group` must make it)."""

    def __init__(self, group=None, slot_bytes=65536):
        from . import _lib
        self.rank, self.world = world(group)
        self.slot_bytes = int(slot_bytes)
        self.handle = ctypes.c_void_p()
        mine = (ctypes.c_ubyte * 64)()
        _lib.check(_lib.lib.vb_comm_create(ctypes.byref(self.handle), self.rank, self.world, self.slot_bytes, mine))
        dev = torch.device('cuda', torch.cuda.current_device())
        on_dev = dist.get_backend(group) == 'nccl'
        t = torch.tensor(list(mine), dtype=torch.uint8, device=dev if on_dev else 'cpu')
        parts = [torch.zeros_like(t) for _ in range(self.world)]
        dist.all_gather(parts, t, group=group)
        blob = b''.join(bytes(p.cpu().tolist()) for p in parts)
        _lib.check(_lib.lib.vb_comm_connect(self.handle, blob))
        dist.barrier(group=group)

    def allreduce_sum_(self, t):
        from . import _lib
        _lib.check(_lib.lib.vb_comm_allreduce_sum_f64(self.handle, _lib.ptr(t), t.numel(), _lib.stream()))
        return t

    def __del__(self):
        try:
            from . import _lib
            if self.handle:
                _lib.lib.vb_comm_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


_comms = {}


def get_communicator(group=None, nbytes=0):
    """The cached communicator of `group` with slots of at least `nbytes` (created collectively on
    first use); None when the process is not distributed or peer memory cannot be mapped on this
    machine (every rank then agrees to use NCCL instead)."""
    if not is_distributed(group) or not torch.cuda.is_available():
        return None
    key = id(group) if group is not None else 0
    comm = _comms.get(key)
    if comm is False:
        return None
    if comm is not None and comm.slot_bytes >= nbytes:
        return comm
    slot = max(65536, (int(nbytes) + 4095) // 4096 * 4096)
    ok = 1
    try:
        comm = Communicator(group, slot)
    except Exception as exc:       # noqa: BLE001  (IPC not permitted, no peer access, ...)
        warnings.warn('viabel_b200: peer-memory communicator unavailable (%s); using NCCL' % exc)
        comm, ok = None, 0
    flag = torch.tensor([ok], dtype=torch.int32, device=torch.device('cuda', torch.cuda.current_device())
                        if dist.get_backend(group) == 'nccl' else 'cpu')
    dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
    if int(flag.item()) == 0:
        _comms[key] = False
        return None
    _comms[key] = comm
    return comm


def allreduce_sum_(t, group=None):
    """In-place sum over ranks (no-op for a single process).  Returns t.  Small contiguous float64 CUDA
    tensors go through the peer-memory communicator (one kernel, rank-ordered and therefore bit-identical
    on every rank); everything else through torch.distributed."""
    if is_distributed(group):
        if t.is_cuda and t.dtype == torch.float64 and t.is_contiguous() and t.numel() * 8 <= 65536:
            comm = get_communicator(group, t.numel() * 8)
            if comm is not None:
                return comm.allreduce_sum_(t)
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return t


def broadcast_seed(seed, group=None):
    """Rank 0's seed on every rank: the sharded objectives need identical base draws everywhere."""
    return int(broadcast_seeds(np.array([int(seed)], dtype=np.uint64), group)[0])


def broadcast_seeds(seeds, group=None):
    """Rank 0's seeds (a uint64 array of values below 2^63) on every rank, in one collective."""
    seeds = np.asarray(seeds, dtype=np.uint64)
    if not is_distributed(group):
        return seeds
    dev = torch.device('cuda', torch.cuda.current_device()) if dist.get_backend(group) == 'nccl' else 'cpu'
    t = torch.as_tensor(seeds.astype(np.int64), device=dev)
    dist.broadcast(t, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
    return t.cpu().numpy().astype(np.uint64)


def allgather_ragged(t, group=None):
    """Concatenate 1-D tensors of different lengths from all ranks (rank order)."""
    if not is_distributed(group):
        return t
    ws = dist.get_world_size(group)
    n = torch.tensor([t.numel()], dtype=torch.int64, device=t.device)
    sizes = [torch.zeros_like(n) for _ in range(ws)]
    dist.all_gather(sizes, n, group=group)
    sizes = [int(s.item()) for s in sizes]
    cap = max(sizes) if sizes else 0
    pad = torch.zeros(cap, dtype=t.dtype, device=t.device)
    pad[:t.numel()] = t
    bufs = [torch.empty_like(pad) for _ in range(ws)]
    dist.all_gather(bufs, pad, group=group)
    return torch.cat([b[:s] for b, s in zip(bufs, sizes)])
