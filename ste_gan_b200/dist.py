"""Data-parallel plumbing: one process per GPU, torch.distributed (NCCL over NVLink 5 / NVSwitch).

The reference is single-process (ste_gan/train.py:545); data parallelism is added here.  It is
exact because no op on the hot path couples samples (no BatchNorm) and every loss is a mean
(train.py:194-196,211,262; time_domain_loss.py:73): averaging the per-shard gradients equals
the global-batch gradient.  Spectral-norm u/v evolve deterministically from (weights, u), so
replicas stay in sync after the initial broadcast.

  training : batch sharded over ranks; ONE exchange step - a bucketed all-reduce (sum) of the flat
             gradient per phase, issued back to front; the 1/world scale is folded into AdamW.
  inference: utterances sharded round-robin; no collective.
"""
from __future__ import annotations

import os
from typing import List, Optional, Tuple

import torch
import torch.distributed as dist


def init_from_env(backend: Optional[str] = None) -> Tuple[int, int, int]:
    """Initialise the default process group from torchrun's env (RANK / WORLD_SIZE / LOCAL_RANK /
    MASTER_ADDR / MASTER_PORT).  Returns (rank, world, local_rank); a no-op (0, 1, 0) without torchrun."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        if backend == "nccl":
            torch.cuda.set_device(local)
            dist.init_process_group(backend, device_id=torch.device("cuda", local))
        else:
            dist.init_process_group(backend)
    return rank, world, local


def shard_range(rank: int, world: int, n: int) -> Tuple[int, int]:
    """Contiguous shard [lo, hi) of n items for `rank` (sizes differ by at most one)."""
    base, rem = divmod(n, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def round_robin(rank: int, world: int, n: int) -> List[int]:
    """Utterance indices served by `rank` for collective-free inference sharding."""
    return list(range(rank, n, world))


class GradReducer:
    """Bucketed all-reduce (SUM) of a flat gradient buffer over the data-parallel group.
    Buckets are issued back to front - the order backward completes them - asynchronously on the
    communicator's stream and waited for before the optimiser kernel, which applies 1/world."""

    def __init__(self, group=None, bucket_mb: float = 32.0, enabled: bool = True):
        """enabled=False: a reducer that does nothing even inside an initialised process group (a single-process reference
        run on one rank; creating the communicator is a collective, so it must not happen on a subset of the ranks)."""
        self.enabled = enabled and dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
        self.group = group
        self.world = dist.get_world_size(group) if self.enabled else 1
        self.bucket = max(1, int(bucket_mb * (1 << 20) // 4))
        # Our own NCCL communicator (ste_gan_b200/nccl.py): all-reduces on explicit streams, capturable inside the CUDA
        # graphs of the train step.  GPU + NCCL backend only; the gloo tests exercise the torch.distributed path.
        self.comm = None
        if self.enabled and torch.cuda.is_available() and dist.get_backend(group) == "nccl":
            from .nccl import NcclComm
            self.comm = NcclComm(group)

    def all_reduce_on(self, flat_slice: torch.Tensor, stream: "torch.cuda.Stream") -> None:
        """SUM all-reduce of a slice of a flat gradient, enqueued on `stream` through the own communicator (works
        eagerly and under CUDA-graph capture; ordering against other streams is the caller's business)."""
        if self.comm is None:
            raise RuntimeError("GradReducer.all_reduce_on needs the own NCCL communicator (CUDA + nccl backend)")
        self.comm.all_reduce(flat_slice, stream)

    @property
    def grad_scale(self) -> float:
        return 1.0 / self.world

    def buckets(self, n: int) -> List[Tuple[int, int]]:
        out, hi = [], n
        while hi > 0:
            lo = max(0, hi - self.bucket)
            out.append((lo, hi))
            hi = lo
        return out

    def all_reduce(self, flat_grad: torch.Tensor) -> None:
        if not self.enabled:
            return
        handles = [dist.all_reduce(flat_grad[lo:hi], op=dist.ReduceOp.SUM, group=self.group, async_op=True)
                   for lo, hi in self.buckets(flat_grad.numel())]
        for h in handles:
            h.wait()

    def all_reduce_async(self, flat_grad: torch.Tensor) -> list:
        """Issue the bucketed all-reduce without waiting; pass the result to wait() before the gradient is consumed."""
        if not self.enabled:
            return []
        return [dist.all_reduce(flat_grad[lo:hi], op=dist.ReduceOp.SUM, group=self.group, async_op=True)
                for lo, hi in self.buckets(flat_grad.numel())]

    @staticmethod
    def wait(handles: list) -> None:
        for h in handles:
            h.wait()

    def broadcast(self, flat: torch.Tensor, src: int = 0) -> None:
        if self.enabled:
            dist.broadcast(flat, src=src, group=self.group)
