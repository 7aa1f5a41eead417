"""Vectorised PPO v1 over the engine's device-resident pieces: the learner of the PPO / DPPO v1 demos
(algorithm/policy_base/Proximal_Policy_Optimization.py, Distributed_PPO.py), restated for N instances on one GPU.

    collect():  as VecPPO2 (K-POLICY -> step kernel -> time-major RolloutBuffer), without the reward normaliser by default
    learn():    R = Monte-Carlo returns (K-RET, every done ends an episode, no bootstrap) with their (sum, sum^2, count)
                -> R_hat = (R - mean) / (std + ret_norm_eps), the statistics all-reduced over a process group ->
                K_epochs full-batch epochs of b200_ppo1_grad (adv = R_hat - V(s) with the current critic, the joint loss
                -min(surr1, surr2) + value_coef mse(V, R_hat) - entropy_coef H) and ONE Adam step over both nets (two
                learning rates, one step count), with a flat gradient all-reduce in between when world > 1

The loss is a restatement checked against float64 autograd of the statement above (tests/test_ppo1_gpu.py), not against
a recording of the reference learner; only the return scan is pinned by a recording (DESIGN 4).  Every constant of the
update is a key of ``ppo_msg``.
"""
from __future__ import annotations

from typing import Optional

import torch

from . import dist as _dist
from . import gae as _gae
from .ppo2 import DEFAULT_PPO_MSG, VecPPO2

# The v1 defaults: Adam eps 1e-8 (set_adam_eps False), no gradient clipping, no learning-rate decay, the critic loss
# weighted by value_coef in the joint loss and the returns normalised with (R - mean) / (std + ret_norm_eps).  Each
# epoch is one full batch: mini_batch_size / using_mini_batch are not read.
DEFAULT_PPO1_MSG = dict(DEFAULT_PPO_MSG, set_adam_eps=False, use_grad_clip=False, use_lr_decay=False, value_coef=0.5,
                        ret_norm_eps=1e-7)


class VecPPO(VecPPO2):
    def __init__(self, env, actor: torch.nn.Module, critic: torch.nn.Module, ppo_msg: Optional[dict] = None,
                 std=None, reward_norm: bool = False, seed: int = 0, group=None, actor_out_act: Optional[str] = None,
                 track_episodes: bool = False):
        """The arguments of :class:`VecPPO2`, with the defaults of ``DEFAULT_PPO1_MSG`` and ``reward_norm`` off (the
        returns are normalised in :meth:`learn`).  The update always runs on K-LEARN: nets it cannot hold raise
        ``B200EnvError``."""
        m = dict(DEFAULT_PPO1_MSG)
        m.update(ppo_msg or {})
        if not float(m['value_coef']) >= 0.0:
            raise ValueError("value_coef must be >= 0")
        super().__init__(env, actor, critic, m, std=std, reward_norm=reward_norm, seed=seed, group=group,
                         actor_out_act=actor_out_act, learner="fused", track_episodes=track_episodes)
        self.value_coef, self.ret_norm_eps = float(m['value_coef']), float(m['ret_norm_eps'])
        T, N = self.buffer.batch_size, self.buffer.n_envs
        dev = env.device
        self._ret_stats = torch.zeros(3, dtype=torch.float64, device=dev)
        self._adv = torch.empty(T, N, dtype=torch.float32, device=dev)
        # the full batch in rollout order: consecutive samples of a tile are consecutive instances of one row, so the
        # observation gathers are coalesced (a keyed permutation would scatter them over the whole rollout)
        self._index = torch.arange(T * N, dtype=torch.int64, device=dev)

    def learn(self) -> dict:
        buf = self.buffer
        world = _dist.dist.get_world_size(self.group) if _dist.dist.is_initialized() else 1
        with torch.no_grad():
            self._ret_stats.zero_()
            ret = _gae.mc_returns(buf.r, buf.done, self.gamma, stats=self._ret_stats)
            _gae.normalize_advantage(ret, self._ret_stats, eps=self.ret_norm_eps, group=self.group)
            B = ret.numel()
            for _ in range(self.K_epochs):
                self.fused.ppo1_grad_step(buf.s, buf.a, buf.a_lp, ret, self._adv, self.value_coef, 0, B,
                                          index=self._index)
                if world > 1:
                    _dist.dist.all_reduce(self.fused.grad, op=_dist.dist.ReduceOp.SUM, group=self.group)
                self.fused.adam_step(1.0 / world)
        self._after_fused_update()
        la, lc = self.fused.loss.tolist()
        return {"actor_loss": la, "critic_loss": lc, "loss": la + lc}
