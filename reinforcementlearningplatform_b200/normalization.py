"""Running mean/std normalisation on device (kernel K-NORM, csrc/norm.cu) -- the vector mirror of
``RunningMeanStd`` / ``Normalization`` (utils/classes.py:626-656).

The reference applies one ``Normalization`` object to every reward (``reward_norm(env.reward)``,
demonstration/PPO2/PPO2-4-CartPoleAngleOnly/train.py:139,210) and, in the UAV envs, to every observation
(``env.current_state_norm(env.current_state, update=True)``, PPO2-4-UavFntsmcParamPos/train.py:291,308).  Each call
there sees ONE sample.  Here a call sees the N samples of one step:

* they enter the statistics together (pairwise Chan merge of ``(count, mean, M2)``) and all N are normalised with the
  merged statistics -- a batch of one sample reproduces the reference's update bit for bit (tests/test_norm.py);
* with ``torch.distributed`` initialised, the per-rank batch statistics (3 x dim doubles) are all-gathered and merged
  in rank order, so every rank holds identical running statistics (``sync=True``);
* ``seq(x)`` feeds ``rows`` samples one after the other (the reference recurrence, bit-exact) for single-instance
  rollouts.

State: ``run[3, dim]`` float64 on device = ``(n, mean, S)``; ``running_ms`` exposes the reference's ``n / mean / S /
std`` names (``std = mean`` while ``n == 1``, sic).
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch

from . import _lib
from ._lib import ptr as _p

EPS = 1e-8  # utils/classes.py:654


def gather_batch_stats(batch: torch.Tensor, out: Optional[torch.Tensor] = None, group=None) -> torch.Tensor:
    """All-gather the per-rank batch statistics ``[1, 3, dim]`` into ``[world, 3, dim]`` (rank order): the only exchange
    of the multi-GPU normaliser, 3 x dim doubles per rank.  Every rank then merges the same list in the same order
    (``b200_norm_merge_apply`` with ``n_batches = world``), so the running statistics stay bit-identical across ranks."""
    import torch.distributed as dist
    w = dist.get_world_size(group)
    if out is None or out.shape[0] != w:
        out = torch.zeros((w,) + tuple(batch.shape[1:]), dtype=batch.dtype, device=batch.device)
    if dist.get_backend(group) == "nccl":
        dist.all_gather_into_tensor(out, batch.contiguous(), group=group)
    else:   # gloo (CPU tests, two ranks on one GPU): all_gather has no CUDA path there -- 3 x dim doubles via the host
        mine = batch.detach().cpu().contiguous()
        parts = [torch.empty_like(mine) for _ in range(w)]
        dist.all_gather(parts, mine, group=group)
        out.copy_(torch.cat(parts, 0).to(out.device))
    return out


class _RunningView:
    """``Normalization.running_ms`` with the reference's attribute names, read from / written to the device state."""

    def __init__(self, owner: "Normalization"):
        self._o = owner

    @property
    def n(self):
        return float(self._o._run[0, 0].item())

    @n.setter
    def n(self, v):
        self._o._run[0].fill_(float(np.asarray(v).reshape(-1)[0]))

    @property
    def mean(self):
        return self._o._run[1].cpu().numpy().copy()

    @mean.setter
    def mean(self, v):
        self._o._run[1].copy_(torch.as_tensor(np.asarray(v, dtype=np.float64).reshape(-1)))

    @property
    def S(self):
        return self._o._run[2].cpu().numpy().copy()

    @S.setter
    def S(self, v):
        self._o._run[2].copy_(torch.as_tensor(np.asarray(v, dtype=np.float64).reshape(-1)))

    @property
    def std(self):
        n, mean, S = self.n, self.mean, self.S
        if n == 1:
            return mean  # `self.std = x` (utils/classes.py:637-639)
        return np.sqrt(S / n) if n > 0 else np.zeros_like(S)

    @std.setter
    def std(self, v):  # derived from (n, S); accepted for load_norm_normalizer_from_file compatibility
        pass


class Normalization:
    """``Normalization(shape)`` of utils/classes.py:646-656 for ``[dim, N]`` field-major batches on one CUDA device."""

    def __init__(self, shape: int, device="cuda", sync: bool = True, group=None):
        self._lib = _lib.load()
        self.dim = int(shape)
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.B200EnvError("the engine has no CPU path: device must be a CUDA device")
        self.sync, self.group = bool(sync), group
        self._run = torch.zeros(3, self.dim, dtype=torch.float64, device=self.device)
        self._run_next = torch.zeros_like(self._run)
        self._batch = torch.zeros(1, 3, self.dim, dtype=torch.float64, device=self.device)
        self._gathered = None
        self._scratch = torch.zeros(self._lib.b200_norm_scratch_bytes(self.dim), dtype=torch.uint8, device=self.device)
        self.running_ms = _RunningView(self)

    # ------------------------------------------------------------------ helpers
    @staticmethod
    def _code(t: torch.Tensor) -> int:
        if t.dtype == torch.float64:
            return _lib.F64
        if t.dtype == torch.float32:
            return _lib.F32
        raise ValueError("normalisation input must be float32 or float64")

    def _world(self) -> int:
        import torch.distributed as dist
        if self.sync and dist.is_available() and dist.is_initialized():
            return dist.get_world_size(self.group)
        return 1

    # ------------------------------------------------------------------ hot call
    def normalize_soa(self, x: torch.Tensor, update: bool = True, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """``x``: contiguous ``[dim, N]`` (or ``[N]`` when dim == 1) CUDA tensor; returns the normalised batch (``out``
        or a new tensor).  One statistics launch + one merge/apply launch; no host synchronisation."""
        if x.dim() == 1:
            x = x.view(1, -1)
        if not (x.is_cuda and x.is_contiguous() and x.shape[0] == self.dim):
            raise ValueError(f"normalize_soa: expected a contiguous CUDA [{self.dim}, N] tensor")
        code, n = self._code(x), x.shape[1]
        y = torch.empty_like(x) if out is None else out.view_as(x)
        with torch.cuda.device(self.device):
            stream = _lib.stream(self.device)
            nb, batch = 0, self._batch
            if update:
                _lib.check(self._lib.b200_norm_batch_stats(code, n, self.dim, _p(x), _p(self._run), _p(self._batch),
                                                           _p(self._scratch), stream), "b200_norm_batch_stats")
                nb = 1
                w = self._world()
                if w > 1:
                    self._gathered = gather_batch_stats(self._batch, self._gathered, self.group)
                    nb, batch = w, self._gathered
            _lib.check(self._lib.b200_norm_merge_apply(code, n, self.dim, _p(x), _p(y), _p(batch), nb, _p(self._run),
                                                       _p(self._run_next), 1 if update else 0, EPS, stream),
                       "b200_norm_merge_apply")
            if update:
                self._run, self._run_next = self._run_next, self._run
        return y

    def normalize_rows(self, x: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """A whole time-major rollout column ``x [T, N]`` of this (one-dimensional) normaliser's feature -- the rewards of
        a rollout -- with row t entering the statistics after rows 0..t-1 and normalised with the statistics after row t:
        what ``T`` calls of ``normalize_soa(x[t], out=x[t])`` do, in three launches (``b200_norm_rows_prefix``).  The
        batch statistics of a row are summed about the row's first sample instead of the running mean, so the result agrees
        with the per-row calls to float64 rounding, not bit for bit.  ``out`` may be ``x``."""
        if self.dim != 1:
            raise ValueError("normalize_rows: a one-dimensional normaliser (reward scaling)")
        if not (x.is_cuda and x.is_contiguous() and x.dim() == 2):
            raise ValueError("normalize_rows: expected a contiguous CUDA [T, N] tensor")
        T, n = x.shape
        code = self._code(x)
        y = torch.empty_like(x) if out is None else out
        if getattr(self, "_rows_T", None) != T:
            self._rows_T = T
            self._rows_batch = torch.zeros(1, 3, T, dtype=torch.float64, device=self.device)
            self._rows_cum = torch.zeros(3, T, dtype=torch.float64, device=self.device)
            self._rows_scratch = torch.zeros(self._lib.b200_norm_scratch_bytes(T), dtype=torch.uint8, device=self.device)
            self._rows_gathered = None
        with torch.cuda.device(self.device):
            stream = _lib.stream(self.device)
            _lib.check(self._lib.b200_norm_batch_stats(code, n, T, _p(x), None, _p(self._rows_batch), _p(self._rows_scratch),
                                                       stream), "b200_norm_batch_stats")
            nb, batch = 1, self._rows_batch
            w = self._world()
            if w > 1:
                self._rows_gathered = gather_batch_stats(self._rows_batch, self._rows_gathered, self.group)
                nb, batch = w, self._rows_gathered
            _lib.check(self._lib.b200_norm_rows_prefix(T, _p(batch), nb, _p(self._run), _p(self._rows_cum), _p(self._run_next),
                                                       stream), "b200_norm_rows_prefix")
            _lib.check(self._lib.b200_norm_merge_apply(code, n, T, _p(x), _p(y), None, 0, _p(self._rows_cum), None, 0, EPS,
                                                       stream), "b200_norm_merge_apply")
            self._run, self._run_next = self._run_next, self._run
        return y

    def __call__(self, x, update: bool = True):
        """Reference call shape: ``x`` is ``[N, dim]`` (or ``[N]`` / a scalar batch for dim == 1); returns the same
        orientation.  ``[dim, N]`` views of the engine's SoA buffers (``env.current_state`` is such a view) are used in
        place, without a transpose copy."""
        if not torch.is_tensor(x):
            x = torch.as_tensor(np.asarray(x, dtype=np.float64), device=self.device)
        if x.dim() == 0:
            x = x.view(1)
        if x.dim() == 1:
            if self.dim == 1:
                return self.normalize_soa(x.contiguous().view(1, -1), update).view(-1)
            return self.normalize_soa(x.contiguous().view(self.dim, 1), update).view(-1)  # one sample of `dim` features
        if x.shape[1] != self.dim:
            raise ValueError(f"expected [N, {self.dim}], got {tuple(x.shape)}")
        soa = x.t() if x.t().is_contiguous() else x.t().contiguous()
        return self.normalize_soa(soa, update).t()

    def seq(self, x: torch.Tensor, update: bool = True) -> torch.Tensor:
        """The reference recurrence over ``rows`` samples fed one by one: ``x`` is ``[dim, rows]`` contiguous."""
        if x.dim() == 1:
            x = x.view(1, -1)
        if not (x.is_cuda and x.is_contiguous() and x.shape[0] == self.dim):
            raise ValueError(f"seq: expected a contiguous CUDA [{self.dim}, rows] tensor")
        y = torch.empty_like(x)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.b200_norm_seq(self._code(x), x.shape[1], self.dim, _p(x), _p(y), _p(self._run),
                                               1 if update else 0, EPS, _lib.stream(self.device)), "b200_norm_seq")
        return y

    # ------------------------------------------------------------------ state
    def state_dict(self) -> dict:
        return {"run": self._run.clone()}

    def load_state_dict(self, sd: dict) -> None:
        self._run.copy_(sd["run"].to(self.device, torch.float64))


def merge_stats_reference(run, batches):
    """Host restatement (numpy float64) of the merge rule of csrc/norm.cu, for tests and offline tooling:
    ``run`` = (n, mean, S) arrays, ``batches`` = iterable of (count, mean, M2)."""
    n, mean, S = (np.array(a, dtype=np.float64, copy=True) for a in run)
    for nb, mb, Mb in batches:
        nb, mb, Mb = (np.asarray(a, dtype=np.float64) for a in (nb, mb, Mb))
        first = n <= 0
        tot = n + nb
        delta = mb - mean
        new_mean = np.where(first, mb, mean + delta * nb / np.where(tot > 0, tot, 1))
        S = np.where(first, Mb, (S + Mb) + delta * (mb - new_mean) * nb)
        n, mean = tot, new_mean
    return n, mean, S
