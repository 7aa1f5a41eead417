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
from .policy import gaussian_head, linear_layers


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
        """``struct b200_mlp`` of net ``k`` (its parameters live in the flat buffer, so the pointers stay valid)."""
        return _lib.mlp(self.layers[k], out_act)


def learn_fits(layers, max_out: int) -> bool:
    """The nets K-LEARN and K-DQN hold (every layer in shared memory): 1..4 linear layers with bias, widths and state_dim
    <= 64, at most ``max_out`` outputs (16 actions for the PPO actor, 64 for a Q-net)."""
    return (1 <= len(layers) <= 4 and all(l.in_features <= 64 and l.out_features <= 64 and l.bias is not None
                                          for l in layers) and layers[-1].out_features <= max_out)


def fused_supported(actor, critic) -> bool:
    """K-LEARN holds every layer in shared memory: <= 4 layers per net, widths and state_dim <= 64, <= 16 actions."""
    critic = linear_layers(critic)
    return learn_fits(linear_layers(actor), 16) and learn_fits(critic, 1) and critic[-1].out_features == 1


class FlatAdam:
    """The parameters of ``nets`` in one flat buffer (:class:`FlatParams`, one Adam segment per net), their gradient and
    Adam moments, and the clip_grad_norm_ + Adam step over all segments in one launch (``b200_adam_step``).  ``lr``: one
    learning rate per net; ``grad_norm``: the gradient norm of every segment at the last step.  The flat buffers are
    allocated here once and never re-bound: the launches hold their addresses."""

    def __init__(self, nets, lr, betas, adam_eps: float, max_grad_norm: float):
        self._lib = _lib.load()
        self.params = FlatParams(nets)
        self.device = self.params.flat.device
        if self.device.type != "cuda":
            raise _lib.B200EnvError("the engine has no CPU path: nets must live on a CUDA device")
        self.lr = [float(x) for x in lr]
        self.adam_eps, self.betas, self.max_grad_norm = float(adam_eps), (float(betas[0]), float(betas[1])), float(max_grad_norm)
        k = len(nets)
        self.grad = torch.zeros(self.params.flat.numel(), dtype=torch.float32, device=self.device)
        self.exp_avg = torch.zeros_like(self.grad)
        self.exp_avg_sq = torch.zeros_like(self.grad)
        self.grad_norm = torch.zeros(k, dtype=torch.float32, device=self.device)
        self.step_count = 0
        # the arguments of b200_adam_step that never change, built once: a small update is bound by its host work
        self._segs = (k, (C.c_int64 * k)(*self.params.net_off), (C.c_int64 * k)(*self.params.net_len))
        self._lr_array = C.c_float * k
        self._bufs = tuple(map(_lib.ptr, (self.params.flat, self.grad, self.exp_avg, self.exp_avg_sq)))
        self._norm_out = _lib.ptr(self.grad_norm)

    def _stream(self):
        return _lib.stream(self.device)

    def adam_step(self, grad_scale: float = 1.0) -> None:
        """clip_grad_norm_ + Adam over every parameter segment (one launch); ``grad_scale`` multiplies the gradient
        first (1 / world size after a summing all-reduce)."""
        self.step_count += 1
        with torch.cuda.device(self.device):
            _lib.check(self._lib.b200_adam_step(
                *self._segs, self._lr_array(*self.lr), *self._bufs, self.step_count, self.betas[0], self.betas[1],
                self.adam_eps, self.max_grad_norm, float(grad_scale), self._norm_out, self._stream()),
                "b200_adam_step")


class FusedPPO2Update(FlatAdam):
    def __init__(self, actor, critic, std, a_min, a_max, actor_out_act: str = "relu", a_lr: float = 1e-4,
                 c_lr: float = 1e-3, adam_eps: float = 1e-5, betas=(0.9, 0.999), max_grad_norm: float = 0.5,
                 eps_clip: float = 0.2, entropy_coef: float = 0.01, group=None):
        if not fused_supported(actor, critic):
            raise _lib.B200EnvError("K-LEARN: nets must have <= 4 layers, widths <= 64, <= 16 actions, 1 value")
        super().__init__([actor, critic], (a_lr, c_lr), betas, adam_eps, max_grad_norm)
        self.out_act, self.a_min, self.a_max, self.std, self.std_vec = gaussian_head(std, a_min, a_max, actor_out_act,
                                                                                     self.device)
        self.eps_clip, self.entropy_coef, self.group = float(eps_clip), float(entropy_coef), group
        self.loss = torch.zeros(2, dtype=torch.float32, device=self.device)
        # the parameters live in the flat buffer from here on, so the descriptors' pointers stay valid
        self.mlps = (self.params.mlp(0, self.out_act), self.params.mlp(1, 0))
        need = int(self._lib.b200_ppo2_workspace_bytes(*map(C.byref, self.mlps)))
        if need == 0:
            raise _lib.B200EnvError("b200_ppo2_workspace_bytes: net not supported by K-LEARN")
        self.workspace = torch.zeros(need, dtype=torch.uint8, device=self.device)

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

    def _args(self, b: _lib.PPO2Batch) -> tuple:
        """The arguments b200_ppo2_grad, b200_ppo1_grad and b200_ppo2_learn share, in their order: the batch, both nets,
        the Gaussian head, the clip range and the entropy coefficient.  Read at every call: ``VecPPO2.set_action_std``
        may have changed the scalar ``std``."""
        p = _lib.ptr
        return (C.byref(b), *map(C.byref, self.mlps), self.std, p(self.std_vec), p(self.a_min), p(self.a_max),
                self.eps_clip, self.entropy_coef)

    def _grads(self) -> tuple:
        """``grad_actor, grad_critic``: the two segments of ``self.grad``."""
        return _lib.ptr(self.grad), C.c_void_p(self.grad.data_ptr() + 4 * self.params.net_off[1])

    def grad_step(self, s, a, a_lp, adv, v_target, first: int, count: int, perm_key: int = 0,
                  index: Optional[torch.Tensor] = None) -> None:
        """Gradients of both mean losses for one mini-batch -> ``self.grad`` ([actor | critic]); losses -> ``self.loss``."""
        b = self._batch(s, a, a_lp, adv, v_target, first, count, perm_key, index)
        p = _lib.ptr
        with torch.cuda.device(self.device):
            _lib.check(self._lib.b200_ppo2_grad(
                *self._args(b), *self._grads(), p(self.loss), p(self.workspace), self.workspace.numel(),
                self._stream()), "b200_ppo2_grad")

    def ppo1_grad_step(self, s, a, a_lp, ret_hat, adv_out, value_coef: float, first: int, count: int, perm_key: int = 0,
                       index: Optional[torch.Tensor] = None, value: Optional[torch.Tensor] = None) -> None:
        """Gradient of the PPO v1 joint loss for one batch (``b200_ppo1_grad``) -> ``self.grad``; ``self.loss`` =
        (actor loss with the entropy term, ``value_coef`` x mse).  ``ret_hat [T, N]``: the normalised returns;
        ``adv_out [T, N]`` receives ``ret_hat - critic(s)`` at the batch's samples, ``value`` (optional) ``critic(s)``."""
        b = self._batch(s, a, a_lp, adv_out, ret_hat, first, count, perm_key, index)
        if value is not None and not (value.is_cuda and value.dtype == torch.float32 and value.is_contiguous()
                                      and tuple(value.shape) == tuple(ret_hat.shape)):
            raise ValueError("K-LEARN: value must be a contiguous CUDA float32 [T, N] tensor")
        p = _lib.ptr
        with torch.cuda.device(self.device):
            _lib.check(self._lib.b200_ppo1_grad(
                *self._args(b), float(value_coef), p(value), *self._grads(), p(self.loss), p(self.workspace),
                self.workspace.numel(), self._stream()), "b200_ppo1_grad")

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
            p = _lib.ptr
            with torch.cuda.device(self.device):
                _lib.check(self._lib.b200_ppo2_learn(
                    *self._args(b), int(k_epochs), int(mini_batch), self.lr[0], self.lr[1], self.betas[0],
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
