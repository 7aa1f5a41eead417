"""Vectorised PPO2 / DPPO2 over the engine's device-resident pieces (SURVEY 8(f)-2,3).

The learner of the reference (algorithm/policy_base/Proximal_Policy_Optimization2.py:17-160, Distributed_PPO2.py) with
the same hyper-parameter dictionary (``ppo_msg``) and the same loss, restructured around N instances on one GPU:

    collect():  row t of the buffer's s --K-POLICY--> a, log_prob  --step kernel--> s_, r, done, flag of row t and the
                policy-facing observation into row t + 1 of s (time-major RolloutBuffer, no copies); after the T steps the
                reward column goes through the running normaliser (K-NORM) row by row in one pass; no host copy
    learn():    V(s), V(s_) by K-POLICY (critic only) -> K-GAE + global advantage normalisation ->
                K_epochs x mini-batches of the clipped-surrogate / entropy / value losses (Adam eps 1e-5, grad-norm clip
                0.5, linear lr decay, as the reference) by K-LEARN (learn.py / csrc/learn.cu: forward + loss + backward
                of both nets in one launch, clip + Adam in a second one, mini-batches drawn by an in-kernel keyed
                permutation) -> with torch.distributed: one flat gradient all-reduce per mini-batch, the synchronous form
                of the DPPO2 gradient push (Distributed_PPO2.py:86-104)

``learner="fused"`` (default whenever the nets fit K-LEARN: layers <= 64 wide, i.e. every PPO2 demo net) runs no torch
library kernel in learn(); ``learner="torch"`` keeps round 1's autograd update on the caller's modules (the 256-wide
DPPO2 demo nets, or as the comparison the tests check K-LEARN against).
"""
from __future__ import annotations

import math
from typing import Optional

import numpy as np
import torch
import torch.nn.functional as F

from . import dist as _dist
from .episodes import EpisodeTracker, evaluate_first_episodes
from .learn import FusedPPO2Update, fused_supported
from .normalization import Normalization
from .policy import GaussianPolicy, gaussian_std, linear_layers
from .rollout import RolloutBuffer

DEFAULT_PPO_MSG = {  # demonstration/PPO2/PPO2-4-CartPoleAngleOnly/train.py:141-158
    'gamma': 0.99, 'K_epochs': 25, 'eps_clip': 0.2, 'buffer_size': 128, 'a_lr': 1e-4, 'c_lr': 1e-3, 'set_adam_eps': True,
    'lmd': 0.95, 'use_adv_norm': True, 'mini_batch_size': 4096, 'entropy_coef': 0.01, 'use_grad_clip': True,
    'use_lr_decay': True, 'max_train_steps': int(5e8), 'using_mini_batch': True,
}


class VecPPO2:
    def __init__(self, env, actor: torch.nn.Module, critic: torch.nn.Module, ppo_msg: Optional[dict] = None,
                 std=None, reward_norm: bool = True, seed: int = 0, group=None, actor_out_act: Optional[str] = None,
                 learner: str = "auto", track_episodes: bool = False):
        """``env``: a vector env built with ``io_dtype=torch.float32, auto_reset=True``; ``actor`` / ``critic``: tanh
        MLPs on ``env.device`` (the reference's PPOActor_Gaussian / PPOCritic shapes, utils/classes.py:529-615);
        ``buffer_size`` of ``ppo_msg`` is the number of time steps T per rollout (T x N transitions per learn()).
        ``actor_out_act``: the head of ``actor.forward`` ("relu", "identity" or "tanh_range"); default: the module's own
        ``out_act`` attribute, else "relu" (PPOActor_Gaussian.forward, utils/classes.py:563-569).  The behaviour policy
        (K-POLICY in ``collect``) and the learner's ``actor(s)`` must use the same head, or the ratios are wrong.
        ``std``: a float or one value per action dimension.
        ``learner``: "fused" (K-LEARN, nets <= 64 wide), "torch" (autograd on the modules) or "auto" (fused if it fits).
        ``track_episodes``: keep per-episode statistics of the raw rewards of every rollout in ``self.episodes``
        (an :class:`EpisodeTracker`; ``self.episodes.summary()`` reads them)."""
        self.env, self.actor, self.critic, self.group = env, actor, critic, group
        m = dict(DEFAULT_PPO_MSG)
        m.update(ppo_msg or {})
        self.msg = m
        self.gamma, self.lmd, self.K_epochs, self.eps_clip = m['gamma'], m['lmd'], m['K_epochs'], m['eps_clip']
        self.buffer = RolloutBuffer(m['buffer_size'], env)
        ar = torch.as_tensor(env.action_range, dtype=torch.float32)
        std = std if std is not None else getattr(actor, 'std', 0.5)
        self.std = torch.as_tensor(std, dtype=torch.float32).reshape(-1).to(env.device)   # [1] or [A]
        out_act = actor_out_act or getattr(actor, 'out_act', 'relu')
        self.policy = GaussianPolicy(linear_layers(actor), linear_layers(critic), ar[:, 0], ar[:, 1],
                                     self.std.cpu().numpy(), device=env.device, seed=seed,
                                     env_index_offset=env.env_index_offset, actor_out_act=out_act)
        self.value_net = GaussianPolicy(None, linear_layers(critic), ar[:, 0], ar[:, 1], 1.0, device=env.device)
        eps = 1e-5 if m['set_adam_eps'] else 1e-8                                   # PPO2.py:50-55
        _dist.broadcast_parameters([actor, critic], 0, group)
        if learner not in ("auto", "fused", "torch"):
            raise ValueError("learner must be 'auto', 'fused' or 'torch'")
        self.fused = None
        if learner == "fused" or (learner == "auto" and fused_supported(actor, critic)):
            self.fused = FusedPPO2Update(actor, critic, self.std, ar[:, 0], ar[:, 1], out_act, a_lr=m['a_lr'],
                                         c_lr=m['c_lr'], adam_eps=eps, max_grad_norm=0.5 if m['use_grad_clip'] else 0.0,
                                         eps_clip=m['eps_clip'], entropy_coef=m['entropy_coef'], group=group)
        else:
            self.optimizer_actor = torch.optim.Adam(actor.parameters(), lr=m['a_lr'], eps=eps)
            self.optimizer_critic = torch.optim.Adam(critic.parameters(), lr=m['c_lr'], eps=eps)
            self.reduce_actor = _dist.FlatGradAllReducer(actor.parameters(), group)
            self.reduce_critic = _dist.FlatGradAllReducer(critic.parameters(), group)
        self._epoch_key = (int(seed) * 0x9E3779B97F4A7C15 + 0x5851F42D4C957F2D) & (2 ** 64 - 1)
        self.reward_norm = Normalization(1, device=env.device, group=group) if reward_norm else None
        self.episodes = EpisodeTracker(env.n_envs, env.device, group=group) if track_episodes else None
        # total_steps counts the env steps of the whole group: every rank decays its learning rates on the same schedule,
        # the one a single process holding all the group's instances would follow
        self.total_steps = 0
        self._group_envs = _dist.agree_sum(env.n_envs, group)
        self._gen = torch.Generator(device=env.device)
        self._gen.manual_seed(seed + 1)

    # ------------------------------------------------------------------ collection (train.py:186-216, vectorised)
    def collect(self) -> float:
        """One rollout of T steps of all N instances; returns the mean raw reward per step (for logging)."""
        env, buf = self.env, self.buffer
        if not env._policy_obs_valid:
            env.reset(True)
            if self.episodes is not None:
                self.episodes.reset_carry()
        # Row t of buf.s is the observation the policy acts on at step t: s[0] is copied once, every step then writes its
        # policy-facing observation straight into the next row (rollout.RolloutBuffer.step, chain_policy_obs).
        buf.s[0].copy_(env._reset_obs)
        if self.reward_norm is not None:
            ms = self.reward_norm.running_ms
            n0, m0 = float(ms.n), float(np.asarray(ms.mean).reshape(-1)[0])
        for t in range(buf.batch_size):
            self.policy(buf.s[t], action=buf.a[t], log_prob=buf.a_lp[t])            # choose_action, PPO2.py:69-76
            buf.step(env, t, buf.a[t], chain_policy_obs=True)                       # step_update + buffer.append
        if self.episodes is not None:
            self.episodes.update(buf.r, buf.done, buf.flag)                         # raw rewards: before K-NORM
        if self.reward_norm is not None:
            # r = reward_norm(env.reward) (:210) for the whole column at once: row t enters the statistics after rows < t
            # and is normalised with the statistics after row t, as the per-step calls did (three launches per rollout)
            self.reward_norm.normalize_rows(buf.r, out=buf.r)
        self.total_steps += buf.batch_size * self._group_envs
        if self.reward_norm is None:
            return float(buf.r.mean())
        # mean raw reward of this rollout from the normaliser's own float64 statistics (n, mean) before and after it (with
        # a process group they are the group's): no per-step reduction of the reward row
        n1, m1 = float(ms.n), float(np.asarray(ms.mean).reshape(-1)[0])
        return (n1 * m1 - n0 * m0) / max(n1 - n0, 1.0)

    def set_action_std(self, std) -> None:
        """Change the exploration std between iterations: ``self.std``, the sampling policy of ``collect()`` and the
        learner's log-probabilities change together.  ``std`` keeps the form the agent was built with: a scalar for a
        scalar std, a vector of the same length for a per-dimension one; anything else raises ``ValueError``."""
        new = np.asarray(std.detach().cpu() if torch.is_tensor(std) else std, dtype=np.float32)
        if new.ndim > 1 or new.size != self.std.numel():
            raise ValueError(f"set_action_std: expected {'a scalar' if self.std.numel() == 1 else f'{self.std.numel()} values'}, "
                             f"got shape {new.shape}")
        if not (np.isfinite(new).all() and (new > 0).all()):
            raise ValueError("set_action_std: std must be finite and positive")
        self.std.copy_(torch.as_tensor(new.reshape(-1), device=self.std.device))
        for holder in (self.policy, self.fused):
            if holder is not None:
                holder.std, holder.std_vec = gaussian_std(new, out=holder.std_vec)

    # ------------------------------------------------------------------ update (PPO2.py:78-170)
    def _log_prob_entropy(self, s, a):
        mean = self.actor(s)
        std = self.std.expand(a.shape[1])
        lp = -((a - mean) ** 2) / (2 * std * std) - torch.log(std) - math.log(math.sqrt(2 * math.pi))
        ent = float((0.5 + 0.5 * math.log(2 * math.pi) + torch.log(std)).sum())           # Normal.entropy().sum(1)
        return lp, ent

    def learn(self) -> dict:
        buf, m = self.buffer, self.msg
        T, N = buf.batch_size, buf.n_envs
        S, A = buf.state_dim, buf.action_dim
        with torch.no_grad():
            # V(s), V(s'): K-POLICY (critic only) row by row -- row t of the time-major buffer IS a [S, N] field-major
            # observation block, so no transposed copy is made
            if getattr(self, "_vs", None) is None or self._vs.shape != (T, N):
                self._vs = torch.empty(T, N, dtype=torch.float32, device=buf.s.device)
                self._vs_next = torch.empty_like(self._vs)
            vs, vs_ = self._vs, self._vs_next
            for t in range(T):
                self.value_net(buf.s[t], value=vs[t])
                self.value_net(buf.s_[t], value=vs_[t])
            adv, v_target = buf.gae(vs, vs_, self.gamma, self.lmd, normalize=m['use_adv_norm'], group=self.group)
            if self.fused is not None:
                return self._learn_fused(adv, v_target)
            s, a, a_lp, _, _, _, _ = buf.to_tensor()
            adv, v_target = adv.reshape(T * N, 1), v_target.reshape(T * N, 1)
            a_lp_sum = a_lp.sum(1, keepdim=True)
        B = T * N
        mb = min(m['mini_batch_size'], B) if m['using_mini_batch'] else B
        # BatchSampler(SubsetRandomSampler(range(B)), mb, drop_last=False) (PPO2.py:104): ceil(B / mb) mini-batches, the last
        # one partial.  Every mini-batch issues gradient all-reduces, so all ranks must run the SAME number of them even
        # when dist.shard() gave them n_local values that differ by one: the count comes from the smallest B of the group
        # and each rank spreads its own B samples evenly over that many batches, as the fused path does
        # (FusedPPO2Update.learn).
        n_mb = _dist.agree_min(-(-B // mb), self.group)
        grouped = _dist.dist.is_initialized() and _dist.dist.get_world_size(self.group) > 1
        bounds = [(B * j) // n_mb for j in range(n_mb + 1)] if grouped else [min(j * mb, B) for j in range(n_mb + 1)]
        last = {}
        for _ in range(self.K_epochs):
            perm = torch.randperm(B, device=s.device, generator=self._gen)
            for j in range(n_mb):
                idx = perm[bounds[j]:bounds[j + 1]]
                lp_now, ent = self._log_prob_entropy(s[idx], a[idx])
                ratios = torch.exp(lp_now.sum(1, keepdim=True) - a_lp_sum[idx])
                surr1 = ratios * adv[idx]
                surr2 = torch.clamp(ratios, 1 - self.eps_clip, 1 + self.eps_clip) * adv[idx]
                actor_loss = (-torch.min(surr1, surr2) - m['entropy_coef'] * ent).mean()
                self.optimizer_actor.zero_grad(set_to_none=False)
                actor_loss.backward()
                self.reduce_actor()
                if m['use_grad_clip']:
                    torch.nn.utils.clip_grad_norm_(self.actor.parameters(), 0.5)
                self.optimizer_actor.step()
                critic_loss = F.mse_loss(v_target[idx], self.critic(s[idx]))
                self.optimizer_critic.zero_grad(set_to_none=False)
                critic_loss.backward()
                self.reduce_critic()
                if m['use_grad_clip']:
                    torch.nn.utils.clip_grad_norm_(self.critic.parameters(), 0.5)
                self.optimizer_critic.step()
                last = {"actor_loss": actor_loss.detach(), "critic_loss": critic_loss.detach()}
        if m['use_lr_decay']:
            self.lr_decay(self.total_steps)
        return {k: float(v) for k, v in last.items()}

    def _learn_fused(self, adv, v_target) -> dict:
        """The K_epochs x mini-batch loop on K-LEARN: mini-batches are consecutive slices of a keyed pseudo-random
        permutation of the T x N samples (one key per epoch: every sample once per epoch, like BatchSampler over
        SubsetRandomSampler, PPO2.py:104)."""
        buf, m = self.buffer, self.msg
        B = buf.batch_size * buf.n_envs
        mb = min(m['mini_batch_size'], B) if m['using_mini_batch'] else B
        n_mb = None
        if _dist.dist.is_initialized() and _dist.dist.get_world_size(self.group) > 1:
            n_mb = _dist.agree_min(-(-B // mb), self.group)
        loss = self.fused.learn(buf.s, buf.a, buf.a_lp, adv, v_target, self.K_epochs, mb, self._epoch_key, n_mb)
        self._epoch_key = (self._epoch_key + self.K_epochs) & (2 ** 64 - 1)
        self._after_fused_update()
        la, lc = loss.tolist()
        return {"actor_loss": la, "critic_loss": lc}

    def _after_fused_update(self) -> None:
        """What follows every K-LEARN update: the packed weights K-POLICY multiplies from are refreshed, then the
        learning rates decay."""
        self.policy.refresh()
        self.value_net.refresh()
        if self.msg['use_lr_decay']:
            self.lr_decay(self.total_steps)

    def lr_decay(self, total_steps):                                                 # PPO2.py:162-171
        if total_steps >= self.msg['max_train_steps']:
            return
        f = 1 - total_steps / self.msg['max_train_steps']
        lr = [max(self.msg['a_lr'] * f, 1e-6), max(self.msg['c_lr'] * f, 1e-6)]
        if self.fused is not None:
            self.fused.lr = lr
            return
        for opt, x in zip((self.optimizer_actor, self.optimizer_critic), lr):
            for g in opt.param_groups:
                g['lr'] = x

    def evaluate(self, obs_soa: torch.Tensor) -> torch.Tensor:
        """actor mean for ``[state_dim, N]`` observations (``agent.evaluate``, PPO2.py:62-66)."""
        zero = torch.zeros(self.policy.action_dim, obs_soa.shape[1], dtype=torch.float32, device=obs_soa.device)
        return self.policy(obs_soa, noise=zero)["action"]

    def evaluate_episodes(self, env, max_steps: int) -> dict:
        """The deterministic policy (``evaluate``: the clamped actor mean) on every instance of ``env`` for one whole
        episode each -- the test episodes of the reference's train loops, vectorised.  ``env``: a separate instance of the
        training env's class built with ``io_dtype=torch.float32, auto_reset=True``; it is reset here and stepped until
        every instance has finished an episode (checked every 64 steps, one host read each) or ``max_steps`` steps have
        run.  Each instance contributes its FIRST episode, so short episodes are not over-represented.  Nothing of the
        agent changes: not the training env, the policy's noise counter, the reward normaliser or the parameters.
        Returns ``ep_return`` (float64, NaN = unfinished), ``ep_length`` and ``ep_flag`` (int32, -1 = unfinished), all
        ``[N]`` device tensors, and the keys of :meth:`EpisodeTracker.summary`."""
        if (env.state_dim, env.action_dim) != (self.policy.state_dim, self.policy.action_dim):
            raise ValueError("evaluate_episodes: env dimensions differ from the policy's")
        zero = torch.zeros(env.action_dim, env.n_envs, dtype=torch.float32, device=env.device)
        action = torch.empty_like(zero)
        log_prob = torch.empty_like(zero)
        act = lambda obs: self.policy(obs, noise=zero, action=action, log_prob=log_prob)
        return evaluate_first_episodes(self.env, env, act, action, max_steps, self.group)


def reference_nets(state_dim: int, action_dim: int, device, init_std: float = 0.5, mean_act: str = "relu"):
    # the Actor carries `out_act` so that VecPPO2 gives K-POLICY the same head as Actor.forward
    """Actor / critic with the layer shapes, tanh activations and orthogonal init of the reference's
    PPOActor_Gaussian / PPOCritic (utils/classes.py:529-615), as plain nn.Modules on ``device``."""
    class Actor(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.fc1, self.fc2 = torch.nn.Linear(state_dim, 64), torch.nn.Linear(64, 64)
            self.fc3, self.mean_layer = torch.nn.Linear(64, 32), torch.nn.Linear(32, action_dim)
            self.std = init_std
            self.out_act = mean_act
            for l, g in ((self.fc1, 1.0), (self.fc2, 1.0), (self.fc3, 1.0), (self.mean_layer, 0.01)):
                torch.nn.init.orthogonal_(l.weight, gain=g)
                torch.nn.init.constant_(l.bias, 0)

        def forward(self, s):
            s = torch.tanh(self.fc3(torch.tanh(self.fc2(torch.tanh(self.fc1(s))))))
            m = self.mean_layer(s)
            return torch.relu(m) if mean_act == "relu" else m

    class Critic(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.fc1, self.fc2, self.fc3 = torch.nn.Linear(state_dim, 64), torch.nn.Linear(64, 32), torch.nn.Linear(32, 1)
            for l in (self.fc1, self.fc2, self.fc3):
                torch.nn.init.orthogonal_(l.weight, gain=1.0)
                torch.nn.init.constant_(l.bias, 0)

        def forward(self, s):
            return self.fc3(torch.tanh(self.fc2(torch.tanh(self.fc1(s)))))

    return Actor().to(device), Critic().to(device)


def dppo2_nets(state_dim: int, action_dim: int, a_min, a_max, device, hidden: int = 256):
    """Actor / critic with the shapes and heads of the DPPO2 demo nets (demonstration/DPPO2/
    DPPO2-4-UGVForwardObstacleAvoidance/train.py:26-107): state-256-256-action with mean = tanh(mean_layer) * gain + off
    (gain = a_max - off, off = (a_min + a_max) / 2, per-dimension init_std = range / 6, :128) and state-256-256-1, tanh
    hidden layers, orthogonal init (gain 0.01 on the mean layer).  ``actor.out_act = "tanh_range"`` tells VecPPO2 which
    head K-POLICY has to apply."""
    a_min_t = torch.as_tensor(a_min, dtype=torch.float32, device=device)
    a_max_t = torch.as_tensor(a_max, dtype=torch.float32, device=device)

    class Actor(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.fc1, self.fc2 = torch.nn.Linear(state_dim, hidden), torch.nn.Linear(hidden, hidden)
            self.mean_layer = torch.nn.Linear(hidden, action_dim)
            self.off = (a_min_t + a_max_t) / 2.0
            self.gain = a_max_t - self.off
            self.std = ((a_max_t - a_min_t) / 2 / 3).cpu().numpy()
            self.out_act = "tanh_range"
            for l, g in ((self.fc1, 1.0), (self.fc2, 1.0), (self.mean_layer, 0.01)):
                torch.nn.init.orthogonal_(l.weight, gain=g)
                torch.nn.init.constant_(l.bias, 0)

        def forward(self, s):
            s = torch.tanh(self.fc2(torch.tanh(self.fc1(s))))
            return torch.tanh(self.mean_layer(s)) * self.gain + self.off

    class Critic(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.fc1, self.fc2, self.fc3 = (torch.nn.Linear(state_dim, hidden), torch.nn.Linear(hidden, hidden),
                                            torch.nn.Linear(hidden, 1))
            for l in (self.fc1, self.fc2, self.fc3):
                torch.nn.init.orthogonal_(l.weight, gain=1.0)
                torch.nn.init.constant_(l.bias, 0)

        def forward(self, s):
            return self.fc3(torch.tanh(self.fc2(torch.tanh(self.fc1(s)))))

    return Actor().to(device), Critic().to(device)
