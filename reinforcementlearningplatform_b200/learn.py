"""The PPO2 / DPPO2 update on device (kernel K-LEARN, csrc/learn.cu).

``FusedPPO2Update`` runs the mini-batch loop of ``Proximal_Policy_Optimization2.learn`` (algorithm/policy_base/
Proximal_Policy_Optimization2.py:102-131) -- actor forward, ``Normal.log_prob``, ratio, clipped surrogate, backward,
``clip_grad_norm_(0.5)``, ``Adam.step``; critic forward, ``mse_loss``, backward, clip, Adam -- with two launches per
mini-batch (``b200_ppo2_grad`` for both nets, ``b200_adam_step`` for both parameter segments) straight from the
time-major device rollout; no torch library kernel runs.  The caller's ``nn.Module`` parameters are re-pointed into ONE
flat float32 buffer ``[actor | critic]`` (``FlatParams``), so the modules keep working (evaluation, checkpoints,
K-POLICY reads the same memory) while gradients, Adam moments and the DPPO2 all-reduce operate on flat buffers.

With ``torch.distributed`` initialised the flat gradient of BOTH nets is summed by one NCCL all-reduce per mini-batch
between the two launches (the synchronous form of the DPPO2 gradient push, Distributed_PPO2.py:86-104; dist.py) and
Adam divides by the world size.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np
import torch

from . import _lib
from .policy import linear_layers


class FlatParams:
    """Moves the ``weight`` / ``bias`` of the given nets' linear layers into one flat float32 buffer (layer order,
    weight before bias: torch's ``parameters()`` order for these nets) and re-points ``p.data`` at views of it."""

    def __init__(self, nets):
        self.layers = [linear_layers(n) for n in nets]
        params = [p for layers in self.layers for lin in layers for p in (lin.weight, lin.bias)]
        dev = params[0].device
        self.net_len = [sum(lin.weight.numel() + lin.bias.numel() for lin in layers) for layers in self.layers]
        self.net_off = [int(x) for x in np.cumsum([0] + self.net_len[:-1])]
        self.flat = torch.empty(sum(self.net_len), dtype=torch.float32, device=dev)
        o = 0
        for p in params:
            n = p.numel()
            self.flat[o:o + n].copy_(p.data.reshape(-1))
            p.data = self.flat[o:o + n].view_as(p)
            o += n

    def mlp(self, k: int, out_act: int) -> _lib.MLP:
        layers = self.layers[k]
        m = _lib.MLP()
        m.n_layers = len(layers)
        m.dims[0] = layers[0].in_features
        for l, lin in enumerate(layers):
            m.dims[l + 1] = lin.out_features
            m.w[l], m.b[l] = lin.weight.data_ptr(), lin.bias.data_ptr()
        m.out_act = out_act
        return m


def fused_supported(actor, critic) -> bool:
    """K-LEARN holds every layer in shared memory: <= 4 layers per net, widths and state_dim <= 64, <= 16 actions."""
    for net in (actor, critic):
        layers = linear_layers(net)
        if not 1 <= len(layers) <= 4:
            return False
        if any(l.in_features > 64 or l.out_features > 64 or l.bias is None for l in layers):
            return False
    return linear_layers(actor)[-1].out_features <= 16 and linear_layers(critic)[-1].out_features == 1


class FusedPPO2Update:
    def __init__(self, actor, critic, std, a_min, a_max, actor_out_act: str = "relu", a_lr: float = 1e-4,
                 c_lr: float = 1e-3, adam_eps: float = 1e-5, betas=(0.9, 0.999), max_grad_norm: float = 0.5,
                 eps_clip: float = 0.2, entropy_coef: float = 0.01, group=None):
        self._lib = _lib.load()
        if not fused_supported(actor, critic):
            raise _lib.B200EnvError("K-LEARN: nets must have <= 4 layers, widths <= 64, <= 16 actions, 1 value")
        self.params = FlatParams([actor, critic])
        self.device = self.params.flat.device
        if self.device.type != "cuda":
            raise _lib.B200EnvError("the engine has no CPU path: nets must live on a CUDA device")
        self.out_act = {"identity": 0, "relu": 1, "tanh_range": 2}[actor_out_act]
        self.a_min = torch.as_tensor(np.asarray(a_min, dtype=np.float32), device=self.device).contiguous()
        self.a_max = torch.as_tensor(np.asarray(a_max, dtype=np.float32), device=self.device).contiguous()
        std_arr = np.asarray(std.detach().cpu() if torch.is_tensor(std) else std, dtype=np.float32).reshape(-1)
        self.std_vec = torch.as_tensor(std_arr, device=self.device).contiguous() if std_arr.size > 1 else None
        self.std = float(std_arr[0])
        self.lr = [float(a_lr), float(c_lr)]
        self.adam_eps, self.betas, self.max_grad_norm = float(adam_eps), (float(betas[0]), float(betas[1])), float(max_grad_norm)
        self.eps_clip, self.entropy_coef, self.group = float(eps_clip), float(entropy_coef), group
        n = self.params.flat.numel()
        self.grad = torch.zeros(n, dtype=torch.float32, device=self.device)
        self.exp_avg = torch.zeros_like(self.grad)
        self.exp_avg_sq = torch.zeros_like(self.grad)
        self.loss = torch.zeros(2, dtype=torch.float32, device=self.device)
        self.grad_norm = torch.zeros(2, dtype=torch.float32, device=self.device)
        self.step_count = 0
        am, cm = self.params.mlp(0, self.out_act), self.params.mlp(1, 0)
        need = int(self._lib.b200_ppo2_workspace_bytes(C.byref(am), C.byref(cm)))
        if need == 0:
            raise _lib.B200EnvError("b200_ppo2_workspace_bytes: net not supported by K-LEARN")
        self.workspace = torch.zeros(need, dtype=torch.uint8, device=self.device)
        self._seg_off = (C.c_int64 * 2)(*self.params.net_off)
        self._seg_len = (C.c_int64 * 2)(*self.params.net_len)

    # ------------------------------------------------------------------ pieces
    def _batch(self, s, a, a_lp, adv, v_target, first, count, perm_key=0, index=None) -> _lib.PPO2Batch:
        T, S, N = s.shape
        for t, shape in ((a, None), (a_lp, a.shape), (adv, (T, N)), (v_target, (T, N))):
            if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and (shape is None or tuple(t.shape) == tuple(shape))):
                raise ValueError("K-LEARN: rollout tensors must be contiguous CUDA float32 [T, dim, N] / [T, N]")
        if not (s.is_contiguous() and s.dtype == torch.float32):
            raise ValueError("K-LEARN: s must be contiguous float32 [T, S, N]")
        b = _lib.PPO2Batch()
        b.T, b.N = T, N
        b.s, b.a, b.a_lp, b.adv, b.v_target = (t.data_ptr() for t in (s, a, a_lp, adv, v_target))
        b.index = None if index is None else index.data_ptr()
        b.first, b.count, b.perm_key = int(first), int(count), int(perm_key) & (2 ** 64 - 1)
        return b

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def grad_step(self, s, a, a_lp, adv, v_target, first: int, count: int, perm_key: int = 0,
                  index: Optional[torch.Tensor] = None) -> None:
        """Gradients of both mean losses for one mini-batch -> ``self.grad`` ([actor | critic]); losses -> ``self.loss``."""
        b = self._batch(s, a, a_lp, adv, v_target, first, count, perm_key, index)
        am, cm = self.params.mlp(0, self.out_act), self.params.mlp(1, 0)
        p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        o = self.params.net_off[1]
        with torch.cuda.device(self.device):
            _lib.check(self._lib.b200_ppo2_grad(
                C.byref(b), C.byref(am), C.byref(cm), self.std, p(self.std_vec), p(self.a_min), p(self.a_max),
                self.eps_clip, self.entropy_coef, p(self.grad), C.c_void_p(self.grad.data_ptr() + 4 * o), p(self.loss),
                p(self.workspace), self.workspace.numel(), self._stream()), "b200_ppo2_grad")

    def ppo1_grad_step(self, s, a, a_lp, ret_hat, adv_out, value_coef: float, first: int, count: int, perm_key: int = 0,
                       index: Optional[torch.Tensor] = None, value: Optional[torch.Tensor] = None) -> None:
        """Gradient of the PPO v1 joint loss for one batch (``b200_ppo1_grad``) -> ``self.grad``; ``self.loss`` =
        (actor loss with the entropy term, ``value_coef`` x mse).  ``ret_hat [T, N]``: the normalised returns;
        ``adv_out [T, N]`` receives ``ret_hat - critic(s)`` at the batch's samples, ``value`` (optional) ``critic(s)``."""
        b = self._batch(s, a, a_lp, adv_out, ret_hat, first, count, perm_key, index)
        if value is not None and not (value.is_cuda and value.dtype == torch.float32 and value.is_contiguous()
                                      and tuple(value.shape) == tuple(ret_hat.shape)):
            raise ValueError("K-LEARN: value must be a contiguous CUDA float32 [T, N] tensor")
        am, cm = self.params.mlp(0, self.out_act), self.params.mlp(1, 0)
        p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        o = self.params.net_off[1]
        with torch.cuda.device(self.device):
            _lib.check(self._lib.b200_ppo1_grad(
                C.byref(b), C.byref(am), C.byref(cm), self.std, p(self.std_vec), p(self.a_min), p(self.a_max),
                self.eps_clip, self.entropy_coef, float(value_coef), p(value), p(self.grad),
                C.c_void_p(self.grad.data_ptr() + 4 * o), p(self.loss), p(self.workspace), self.workspace.numel(),
                self._stream()), "b200_ppo1_grad")

    def adam_step(self, grad_scale: float = 1.0) -> None:
        """clip_grad_norm_ + Adam over both parameter segments (one launch)."""
        self.step_count += 1
        lr = (C.c_float * 2)(*self.lr)
        p = lambda t: C.c_void_p(t.data_ptr())
        with torch.cuda.device(self.device):
            _lib.check(self._lib.b200_adam_step(
                2, self._seg_off, self._seg_len, lr, p(self.params.flat), p(self.grad), p(self.exp_avg), p(self.exp_avg_sq),
                self.step_count, self.betas[0], self.betas[1], self.adam_eps, self.max_grad_norm, float(grad_scale),
                p(self.grad_norm), self._stream()), "b200_adam_step")

    # ------------------------------------------------------------------ the loop
    def learn(self, s, a, a_lp, adv, v_target, k_epochs: int, mini_batch: int, perm_key: int, n_mb: Optional[int] = None):
        """K_epochs x ceil(B / mini_batch) mini-batches over the rollout ``s [T, S, N]`` ... ``v_target [T, N]``.
        Single process: the whole loop is one C call (no host work between mini-batches).  With a process group: one
        flat all-reduce per mini-batch between the gradient and the Adam launch; ``n_mb`` (agreed over ranks) fixes the
        number of mini-batches per epoch so that every rank issues the same collectives."""
        import torch.distributed as dist
        T, _, N = s.shape
        B = T * N
        world = dist.get_world_size(self.group) if dist.is_available() and dist.is_initialized() else 1
        if world == 1 and n_mb is None:
            b = self._batch(s, a, a_lp, adv, v_target, 0, B, perm_key)
            am, cm = self.params.mlp(0, self.out_act), self.params.mlp(1, 0)
            p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
            with torch.cuda.device(self.device):
                _lib.check(self._lib.b200_ppo2_learn(
                    C.byref(b), C.byref(am), C.byref(cm), self.std, p(self.std_vec), p(self.a_min), p(self.a_max),
                    self.eps_clip, self.entropy_coef, int(k_epochs), int(mini_batch), self.lr[0], self.lr[1], self.betas[0],
                    self.betas[1], self.adam_eps, self.max_grad_norm, self.step_count + 1, p(self.params.flat), p(self.grad),
                    p(self.exp_avg), p(self.exp_avg_sq), p(self.loss), p(self.workspace), self.workspace.numel(),
                    self._stream()), "b200_ppo2_learn")
            self.step_count += int(k_epochs) * (-(-B // int(mini_batch)))
            return self.loss
        n_mb = n_mb or -(-B // int(mini_batch))
        bounds = [(B * j) // n_mb for j in range(n_mb + 1)]
        for e in range(int(k_epochs)):
            for j in range(n_mb):
                self.grad_step(s, a, a_lp, adv, v_target, bounds[j], bounds[j + 1] - bounds[j], perm_key + e)
                if world > 1:
                    dist.all_reduce(self.grad, op=dist.ReduceOp.SUM, group=self.group)
                self.adam_step(1.0 / world)
        return self.loss
