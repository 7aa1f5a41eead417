"""GAE reverse scan + advantage normalisation on device (kernel K-GAE, csrc/gae.cu).

Replaces ``Proximal_Policy_Optimization2.learn`` lines 88-100 (and ``Distributed_PPO2.Worker.learn`` 59-71) for a
time-major ``[T, N]`` rollout: every column is one env instance.  With ``torch.distributed`` initialised the
normalisation statistics ``(sum adv, sum adv^2, count)`` are all-reduced (3 doubles over NCCL) so that every rank
normalises with the GLOBAL mean / unbiased std, the multi-GPU analogue of ``adv.mean()`` / ``adv.std()``.
"""
from __future__ import annotations

import torch

from . import _lib
from ._lib import ptr as _p


def _scratch(N: int, device) -> torch.Tensor:
    """Per-block partial sums of the advantage statistics (fixed-order reduction: bit-reproducible runs)."""
    return torch.empty(max(1, int(_lib.load().b200_gae_scratch_bytes(N)) // 8), dtype=torch.float64, device=device)


def gae(r, vs, vs_next, done, success, gamma: float, lmd: float, acc_mode: int = 0, stats: torch.Tensor = None):
    """adv, v_target, stats = gae(...).  All inputs: CUDA float32 ``[T, N]`` contiguous (done / success as 0.0 / 1.0).
    acc_mode 0 = float32 sequential (bit-identical to the reference loop under numpy >= 2), 1 = float64 carry."""
    lib = _lib.load()
    ts = [r, vs, vs_next, done, success]
    for t in ts:
        if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and t.shape == r.shape and t.dim() == 2):
            raise ValueError("gae: inputs must be contiguous CUDA float32 tensors of one [T, N] shape")
    T, N = r.shape
    adv = torch.empty_like(r)
    vt = torch.empty_like(r)
    if stats is None:
        stats = torch.zeros(3, dtype=torch.float64, device=r.device)
    with torch.cuda.device(r.device):
        scr = _scratch(N, r.device)
        _lib.check(lib.b200_gae(T, N, *[_p(t) for t in ts], float(gamma), float(lmd), int(acc_mode), _p(adv), _p(vt),
                                _p(stats), _p(scr), scr.numel() * 8, _lib.stream(r.device)), "b200_gae")
    return adv, vt, stats


def gae_flags(r, vs, vs_next, done_u8, flag_i32, timeout_flag: int, gamma: float, lmd: float, acc_mode: int = 0,
              stats: torch.Tensor = None):
    """:func:`gae` over a device-resident rollout (``rollout.RolloutBuffer``): ``done_u8`` / ``flag_i32`` are the
    ``is_terminal`` / ``terminal_flag`` columns the step kernel wrote, success = done and flag != timeout_flag."""
    lib = _lib.load()
    for t in (r, vs, vs_next):
        if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and t.shape == r.shape and t.dim() == 2):
            raise ValueError("gae_flags: r, vs, vs_next must be contiguous CUDA float32 tensors of one [T, N] shape")
    if not (done_u8.dtype == torch.uint8 and flag_i32.dtype == torch.int32 and done_u8.shape == r.shape
            and flag_i32.shape == r.shape and done_u8.is_contiguous() and flag_i32.is_contiguous()):
        raise ValueError("gae_flags: done must be uint8 and flag int32, contiguous [T, N]")
    T, N = r.shape
    adv = torch.empty_like(r)
    vt = torch.empty_like(r)
    if stats is None:
        stats = torch.zeros(3, dtype=torch.float64, device=r.device)
    with torch.cuda.device(r.device):
        scr = _scratch(N, r.device)
        _lib.check(lib.b200_gae_flags(T, N, _p(r), _p(vs), _p(vs_next), _p(done_u8), _p(flag_i32), int(timeout_flag),
                                      float(gamma), float(lmd), int(acc_mode), _p(adv), _p(vt), _p(stats), _p(scr),
                                      scr.numel() * 8, _lib.stream(r.device)), "b200_gae_flags")
    return adv, vt, stats


def normalize_advantage(adv: torch.Tensor, stats: torch.Tensor, eps: float = 1e-5, group=None) -> torch.Tensor:
    """In place ``adv <- (adv - mean) / (std + eps)`` (PPO2.py:99-100); ``stats`` from :func:`gae`.  If a process group
    is initialised the 3 statistics are summed over ranks first (global normalisation)."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM, group=group)
    lib = _lib.load()
    with torch.cuda.device(adv.device):
        _lib.check(lib.b200_adv_normalize(adv.numel(), _p(adv), _p(stats), float(eps), _lib.stream(adv.device)),
                   "b200_adv_normalize")
    return adv


def mc_returns(r: torch.Tensor, done_u8: torch.Tensor, gamma: float, stats: torch.Tensor = None) -> torch.Tensor:
    """Monte-Carlo returns of PPO / DPPO v1 (Proximal_Policy_Optimization.py:113-119) over a time-major ``[T, N]``
    rollout: ``r`` float64 (like ``RolloutBuffer.r``) or float32, ``done_u8`` uint8; float64 recurrence, float32 out.
    ``stats``: a CUDA float64 ``[3]`` tensor that is INCREMENTED by (sum R, sum R^2, T * N), summed in a fixed order --
    what :func:`normalize_advantage` reads to normalise the returns."""
    if not (r.is_cuda and r.dim() == 2 and r.is_contiguous() and r.dtype in (torch.float32, torch.float64)):
        raise ValueError("mc_returns: r must be a contiguous CUDA [T, N] float32/float64 tensor")
    if not (done_u8.dtype == torch.uint8 and done_u8.shape == r.shape and done_u8.is_contiguous()):
        raise ValueError("mc_returns: done must be a contiguous uint8 [T, N] tensor")
    if stats is not None and not (stats.is_cuda and stats.dtype == torch.float64 and stats.numel() == 3
                                  and stats.is_contiguous()):
        raise ValueError("mc_returns: stats must be a contiguous CUDA float64 tensor of 3 elements")
    T, N = r.shape
    out = torch.empty(T, N, dtype=torch.float32, device=r.device)
    dt = _lib.F64 if r.dtype == torch.float64 else _lib.F32
    with torch.cuda.device(r.device):
        stream = _lib.stream(r.device)
        if stats is None:
            _lib.check(_lib.load().b200_mc_returns(dt, T, N, _p(r), _p(done_u8), float(gamma), _p(out), stream),
                       "b200_mc_returns")
        else:
            scr = _scratch(N, r.device)
            _lib.check(_lib.load().b200_mc_returns_stats(dt, T, N, _p(r), _p(done_u8), float(gamma), _p(out), _p(stats),
                                                         _p(scr), scr.numel() * 8, stream), "b200_mc_returns_stats")
    return out
