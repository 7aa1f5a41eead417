"""Multi-GPU plumbing: one process per GPU, env instances sharded independently (SURVEY.md section 8e).

* Stepping needs NO collective: rank r owns the contiguous block of instances [r * n_local, (r + 1) * n_local) and
  passes ``env_index_offset = r * n_local`` to its VecEnv, so the in-kernel Philox reset draws depend only on the
  GLOBAL instance index -- trajectories are invariant to the number of GPUs.
* Two real exchange steps exist, both tiny and latency-bound on NVLink 5 / NVSwitch:
    1. global advantage-normalisation statistics: 3 doubles (gae.normalize_advantage);
    2. the DPPO2 gradient hand-off.  The reference pushes each worker's gradients into shared-memory global nets and
       steps an unlocked SharedAdam (demonstration/DPPO2/*/Distributed_PPO2.py:86-104, utils/classes.py:676-691 --
       Hogwild).  Here every rank computes its gradients on its own rollouts and ``FlatGradAllReducer`` averages
       them with ONE ncclAllReduce over a persistent flat fp32 buffer (154 k parameters = 0.6 MB for the 41-256-256
       nets), turning the asynchronous scheme into synchronous data parallelism -- a deliberate semantic change
       (parity is defined on env trajectories and GAE, not on learning curves).
"""
from __future__ import annotations

import os
from typing import Iterable, Tuple

import torch
import torch.distributed as dist


def init_from_env(backend: str = None) -> Tuple[int, int, int]:
    """Initialise torch.distributed from RANK / WORLD_SIZE / LOCAL_RANK / MASTER_* (torchrun).  Returns
    (rank, world, local_rank).  Single-process runs return (0, 1, 0) without creating a group."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and not dist.is_initialized():
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        kw = {}
        if backend == "nccl":
            torch.cuda.set_device(local)
            kw["device_id"] = torch.device("cuda", local)
        dist.init_process_group(backend, **kw)
    return rank, world, local


def shard(n_total: int, rank: int, world: int) -> Tuple[int, int]:
    """(n_local, env_index_offset) of this rank: contiguous blocks, the first n_total % world ranks get one more."""
    base, rem = divmod(int(n_total), int(world))
    n_local = base + (1 if rank < rem else 0)
    offset = rank * base + min(rank, rem)
    return n_local, offset


class FlatGradAllReducer:
    """Averages the gradients of `params` over all ranks with a single all-reduce of one flat buffer."""

    def __init__(self, params: Iterable[torch.nn.Parameter], group=None):
        self.params = [p for p in params if p.requires_grad]
        self.group = group
        n = sum(p.numel() for p in self.params)
        dev = self.params[0].device if self.params else torch.device("cpu")
        self.flat = torch.zeros(n, dtype=torch.float32, device=dev)
        self.views = []
        o = 0
        for p in self.params:
            self.views.append(self.flat[o:o + p.numel()].view_as(p))
            o += p.numel()

    @property
    def nbytes(self) -> int:
        return self.flat.numel() * 4

    def __call__(self) -> None:
        world = dist.get_world_size(self.group) if dist.is_initialized() else 1
        if world == 1:
            return
        for p, v in zip(self.params, self.views):
            if p.grad is None:
                v.zero_()
            else:
                v.copy_(p.grad)
        dist.all_reduce(self.flat, op=dist.ReduceOp.SUM, group=self.group)
        self.flat.div_(world)
        for p, v in zip(self.params, self.views):
            if p.grad is None:
                p.grad = v.clone()
            else:
                p.grad.copy_(v)


def broadcast_parameters(modules: Iterable[torch.nn.Module], src: int = 0, group=None) -> None:
    """Rank `src`'s weights to every rank (the reference's workers start from the shared global nets)."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return
    for m in modules:
        for t in list(m.parameters()) + list(m.buffers()):
            dist.broadcast(t.data, src=src, group=group)


def allreduce_stats(stats: torch.Tensor, group=None) -> torch.Tensor:
    """Sum (sum adv, sum adv^2, count) over ranks in place: the 3-double exchange of the global advantage norm."""
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM, group=group)
    return stats


def agree_sum(value: int, group=None) -> int:
    """The sum of an integer over the ranks of ``group`` (the value itself without torch.distributed): e.g. the group's
    instance count, so that counters derived from it are the same on every rank."""
    return _agree(value, group, dist.ReduceOp.SUM) if dist.is_available() else int(value)


def agree_min(value: int, group=None) -> int:
    """The minimum of an integer over the ranks of ``group`` (the value itself without torch.distributed).  Used to agree
    on loop trip counts that contain collectives: ranks whose shard sizes differ by one must not issue different numbers
    of all-reduces (NCCL would deadlock)."""
    return _agree(value, group, dist.ReduceOp.MIN) if dist.is_available() else int(value)


def _agree(value: int, group, op) -> int:
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return int(value)
    dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend(group) == "nccl" else torch.device("cpu")
    t = torch.tensor([int(value)], dtype=torch.int64, device=dev)
    dist.all_reduce(t, op=op, group=group)
    return int(t.item())
