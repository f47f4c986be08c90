"""Data parallelism over molecules (SURVEY.md section 8e): one process per GPU, each rank trains on its own
mini-batch shard (BatchNorm statistics, recon and contrastive losses stay per rank, exactly as if the reference ran at
the per-rank batch size); the only exchange is ONE all-reduce of the flat gradient buffer per step (NCCL over
NVLink 5 / NVSwitch), followed by the fused Adam with grad_scale = 1 / world_size."""
from __future__ import annotations

import os

import torch
import torch.distributed as dist


def init_from_env(backend: str | None = None):
    """Initialise torch.distributed from RANK / WORLD_SIZE / LOCAL_RANK / MASTER_* (torchrun).  Returns
    (rank, local_rank, world)."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and not dist.is_initialized():
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        kw = {}
        if backend == "nccl":
            torch.cuda.set_device(local_rank)
            kw["device_id"] = torch.device("cuda", local_rank)
        dist.init_process_group(backend, **kw)
    return rank, local_rank, world


def shard_range(num_graphs: int, rank: int, world: int):
    """Contiguous shard [lo, hi) of a global batch: rank r takes graphs r*B_local .. (r+1)*B_local (the remainder is
    spread over the first ranks)."""
    base, rem = divmod(num_graphs, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def rank_world():
    """(rank, world) of the initialised process group; (0, 1) without one."""
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def round_robin_batches(num_items: int, batch_size: int, rank: int, world: int):
    """Whole-batch shard for evaluation: the [lo, hi) item ranges of batches rank, rank + world, rank + 2 world, ... of
    the single-process batch list (the last batch may be short).  The union over the ranks is that batch list, so every
    item is evaluated exactly once whatever ``num_items`` is."""
    starts = range(rank * batch_size, num_items, world * batch_size)
    return [(lo, min(lo + batch_size, num_items)) for lo in starts]


def mean_over_ranks(sums, count: int, device=None):
    """Per-batch means over the union of every rank's batches: ``sums`` are this rank's sums of per-batch values,
    ``count`` its number of batches.  One all-reduce (float64) of the sums and the count; every rank gets the same
    floats back."""
    _, world = rank_world()
    if world == 1:
        return [float(s) / max(count, 1) for s in sums]
    t = torch.tensor([float(s) for s in sums] + [float(count)], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    vals = t.tolist()
    return [s / max(vals[-1], 1.0) for s in vals[:-1]]


@torch.no_grad()
def average_bn_buffers_(module: torch.nn.Module):
    """All-reduce-average ``running_mean`` / ``running_var`` of every BatchNorm in ``module`` across the ranks, in place:
    the buffers of the GIN engine path are views into the engine's ``bn_running`` and must keep aliasing it.  BatchNorm
    batch statistics stay per rank during training, so the running estimates drift apart; averaging them before an
    evaluation or a checkpoint keeps the replicas identical.  ``num_batches_tracked`` is left alone (equal on every rank
    when every rank runs the same number of batches)."""
    _, world = rank_world()
    if world == 1:
        return
    bufs = [b for m in module.modules() if isinstance(m, torch.nn.modules.batchnorm._BatchNorm) and m.track_running_stats
            for b in (m.running_mean, m.running_var)]
    if not bufs:
        return
    flat = torch.cat([b.reshape(-1) for b in bufs])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM)
    flat /= world
    off = 0
    for b in bufs:
        b.copy_(flat[off:off + b.numel()].view_as(b))
        off += b.numel()


def allreduce_grads_(flat_grads: torch.Tensor, world: int) -> float:
    """Sum-all-reduce the flat gradient buffer in place; returns the scale the optimiser applies (1/world)."""
    if world > 1:
        dist.all_reduce(flat_grads, op=dist.ReduceOp.SUM)
    return 1.0 / world


def broadcast_params_(flat_params: torch.Tensor, src: int = 0):
    if dist.is_initialized() and dist.get_world_size() > 1:
        dist.broadcast(flat_params, src)


class _RawCuda:
    """Zero-copy torch view of a raw device allocation (memory the library cudaMalloc'ed for CUDA IPC)."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (int(ptr), False), "version": 2}


def raw_cuda_tensor(ptr: int, nbytes: int, device) -> torch.Tensor:
    return torch.as_tensor(_RawCuda(ptr, nbytes), device=device)


class PeerAllreduce:
    """Gradient exchange fused with Adam over NVLink peer memory (csrc/peer_kernels.cu): every rank allocates two flat
    gradient buffers (step parity) and a flag array through the library, exchanges their CUDA IPC handles over the
    process group and maps the peers' buffers.  ``grads(seq)`` is the buffer the backward pass of step ``seq`` must
    write; ``step(...)`` launches the one fused kernel."""

    def __init__(self, lib, n_floats: int, device, group=None):
        import ctypes
        self.lib, self.device, self.n = lib, torch.device(device), int(n_floats)
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        if self.world > 16:
            raise RuntimeError("PeerAllreduce supports up to 16 ranks on one node")
        from . import _lib as L

        def alloc(nbytes):
            ptr = ctypes.c_void_p()
            h = ctypes.create_string_buffer(64)
            L.check(lib.scgib_peer_alloc(nbytes, ctypes.byref(ptr), h), "peer_alloc")
            return ptr.value, h.raw

        gbytes = self.n * 4
        mine = [alloc(gbytes), alloc(gbytes), alloc(256)]          # grads parity 0, parity 1, flags
        self._own = [p for p, _ in mine]
        handles = [None] * self.world
        dist.all_gather_object(handles, [h for _, h in mine], group=group)
        self._opened = []
        self._ptrs = [[0] * self.world for _ in range(3)]
        for r in range(self.world):
            for k in range(3):
                if r == self.rank:
                    self._ptrs[k][r] = mine[k][0]
                else:
                    ptr = ctypes.c_void_p()
                    L.check(lib.scgib_peer_open(handles[r][k], ctypes.byref(ptr)), "peer_open")
                    self._ptrs[k][r] = ptr.value
                    self._opened.append(ptr.value)
        self._arr = [(ctypes.c_void_p * self.world)(*self._ptrs[k]) for k in range(3)]
        self._grads = [raw_cuda_tensor(mine[k][0], gbytes, self.device).view(torch.float32) for k in range(2)]
        self.seq = 0
        dist.barrier(group=group)                                   # every rank has mapped every buffer

    def grads(self, seq: int) -> torch.Tensor:
        return self._grads[seq & 1]

    def step(self, params, exp_avg, exp_avg_sq, seq, adam_step, lr, betas, eps, weight_decay, stream):
        from . import _lib as L
        L.check(self.lib.scgib_allreduce_adam_f32(L.ptr(params), L.ptr(exp_avg), L.ptr(exp_avg_sq), self.n,
                                                  self._arr[seq & 1], self._arr[2], self.rank, self.world, seq, adam_step,
                                                  lr, betas[0], betas[1], eps, weight_decay, stream), "allreduce_adam")
