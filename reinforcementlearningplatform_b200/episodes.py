"""Episode returns, lengths and end reasons on device (kernel K-EPISODE, csrc/episodes.cu).

The reference's train loops judge a policy by the reward summed over each episode, by how long episodes last and by why
they end (``terminal_flag``), and test the deterministic policy on whole episodes.  ``EpisodeTracker`` does that
bookkeeping for N auto-reset instances at once: it scans the ``[T, N]`` reward / done / flag columns of a rollout (or the
``[N]`` buffers of one step), carries the episode in progress of every instance from one call to the next, keeps the
last finished episode of every instance, and increments float64 statistics (count, return and length sums and sums of
squares, a histogram of the terminal flag) that are reduced in a fixed order on the device.  Reading them is one host
copy; with ``torch.distributed`` initialised they are summed over ranks first.
"""
from __future__ import annotations

import ctypes as C
import math

import torch

from . import _lib

STATS = 22                # B200_EPISODE_STATS (include/b200env.h)
FLAG_BINS = 16            # flags 0 .. 15 have a bin each; index 16 of flag_counts counts every other flag


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class EpisodeTracker:
    def __init__(self, n_envs: int, device, first_only: bool = False, group=None):
        """``first_only``: every instance contributes its first finished episode only (evaluation); later episodes are
        neither recorded nor counted.  ``group``: the process group ``summary()`` sums the statistics over."""
        self.n_envs, self.device = int(n_envs), torch.device(device)
        if self.device.type != "cuda":
            raise _lib.B200EnvError("the engine has no CPU path: device must be a CUDA device")
        if self.device.index is None:          # "cuda" -> "cuda:k", the device tensors report
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.first_only, self.group = bool(first_only), group
        self._lib = _lib.load()
        N, dev = self.n_envs, self.device
        self.acc_return = torch.zeros(N, dtype=torch.float64, device=dev)    # carry: the episode in progress
        self.acc_length = torch.zeros(N, dtype=torch.int32, device=dev)
        self.ep_return = torch.empty(N, dtype=torch.float64, device=dev)     # the last finished episode
        self.ep_length = torch.empty(N, dtype=torch.int32, device=dev)
        self.ep_flag = torch.empty(N, dtype=torch.int32, device=dev)
        self.stats = torch.zeros(STATS, dtype=torch.float64, device=dev)
        self._scratch = torch.empty(max(1, int(self._lib.b200_episode_scratch_bytes(N)) // 8), dtype=torch.float64,
                                    device=dev)
        self.reset()

    def reset_carry(self) -> None:
        """Forget the episodes in progress (call when the env itself is reset)."""
        self.acc_return.zero_()
        self.acc_length.zero_()

    def reset_stats(self) -> None:
        """Start new statistics (e.g. one log row per rollout); carry and records are kept."""
        self.stats.zero_()

    def reset(self) -> None:
        """Zero the carry and the statistics; no instance has a finished episode (return NaN, length and flag -1)."""
        self.reset_carry()
        self.ep_return.fill_(math.nan)
        self.ep_length.fill_(-1)
        self.ep_flag.fill_(-1)
        self.reset_stats()

    def update(self, r: torch.Tensor, done: torch.Tensor, flag: torch.Tensor) -> None:
        """Scan ``T`` rows of rewards (float32 or float64), ``done`` (uint8 or bool) and ``flag`` (int32), each ``[T, N]``
        time-major or ``[N]`` for one step, in ascending t.  Every done row ends an episode (auto-reset envs)."""
        if done.dtype == torch.bool:
            done = done.view(torch.uint8)
        shape = tuple(r.shape)
        if not (len(shape) in (1, 2) and shape[-1] == self.n_envs):
            raise ValueError(f"update: expected [T, {self.n_envs}] or [{self.n_envs}] tensors, got {shape}")
        if r.dtype not in (torch.float32, torch.float64) or done.dtype != torch.uint8 or flag.dtype != torch.int32:
            raise ValueError("update: r must be float32 / float64, done uint8 / bool and flag int32")
        for t in (r, done, flag):
            if tuple(t.shape) != shape or not t.is_contiguous() or t.device != self.device:
                raise ValueError(f"update: r, done and flag must be contiguous tensors of one shape on {self.device}")
        T = shape[0] if len(shape) == 2 else 1
        with torch.cuda.device(self.device):
            stream = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
            _lib.check(self._lib.b200_episode_scan(
                _lib.F64 if r.dtype == torch.float64 else _lib.F32, T, self.n_envs, _p(r), _p(done), _p(flag),
                _p(self.acc_return), _p(self.acc_length), _p(self.ep_return), _p(self.ep_length), _p(self.ep_flag),
                int(self.first_only), _p(self.stats), _p(self._scratch), self._scratch.numel() * 8, stream),
                "b200_episode_scan")

    def finished(self) -> torch.Tensor:
        """bool ``[N]``: the instances that have finished at least one episode since ``reset()``."""
        return self.ep_flag != -1

    def summary(self) -> dict:
        """The statistics of every episode counted since ``reset()`` or ``reset_stats()`` (summed over the ranks of the process group, if
        one is initialised): ``episodes``, ``mean_return``, ``std_return``, ``mean_length``, ``std_length`` (population
        std; NaN without episodes) and ``flag_counts`` (17 ints: episodes ending with flag 0 .. 15, then any other)."""
        import torch.distributed as dist
        st = self.stats
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(self.group) > 1:
            # NCCL reduces device tensors; gloo takes the 22 doubles through the host
            st = st.clone() if dist.get_backend(self.group) == "nccl" else st.cpu()
            dist.all_reduce(st, op=dist.ReduceOp.SUM, group=self.group)
        v = st.tolist()
        n = v[0]
        mean = lambda k: v[k] / n if n > 0 else math.nan
        std = lambda k: math.sqrt(max(v[k + 1] / n - mean(k) ** 2, 0.0)) if n > 0 else math.nan
        return {"episodes": int(n), "mean_return": mean(1), "std_return": std(1), "mean_length": mean(3),
                "std_length": std(3), "flag_counts": [int(c) for c in v[5:5 + FLAG_BINS + 1]]}
