"""Vectorised DQN / Double DQN on the device (K-DQN, csrc/learn.cu): the learner family of the reference's DQN demos
(algorithm/value_base/{DQN,Double_DQN}.py) for the discrete-action env FlightAttitudeSimulatorDiscrete, restated for N
instances on one GPU.

    collect(steps):  per step, b200_dqn_act (epsilon-greedy Q forward, one launch) writes the action index into the replay
                     ring and the action value into the env's action buffer, and the step kernel writes s_, r, done and
                     flag into the same ring row and the next policy observation straight into the next row's s
    learn(updates):  per update, b200_dqn_grad (target, gradient, fixed-order reduction) and b200_adam_step; the target
                     net is a second flat parameter buffer, refreshed by a device copy every target_replace_iter updates

No torch library kernel runs in either loop, and there is no torch fallback: a net K-DQN cannot hold raises.  The update
is this project's statement of the algorithm (checked against float64 autograd of that statement,
tests/test_dqn_gpu.py), not a recording of the reference learner; every constant is a key of ``dqn_msg``.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Optional

import torch

from . import _lib
from . import dist as _dist
from .episodes import EpisodeTracker, evaluate_first_episodes
from .learn import FlatAdam, learn_fits
from .policy import linear_layers

DEFAULT_DQN_MSG = {
    'memory_capacity': 64,       # R rows of the replay ring; R - 1 of them hold sampleable transitions
    'batch_size': 4096,          # samples per update, drawn with replacement
    'gamma': 0.99,
    'lr': 1e-3,
    'betas': (0.9, 0.999),
    'adam_eps': 1e-8,
    'max_grad_norm': 0.0,        # <= 0: no clipping
    'target_replace_iter': 100,  # the target net is copied from the online net before updates 0, T, 2T, ...
    'learn_start': 8,            # learn() does nothing until this many ring rows are valid
    'double_dqn': False,
}

_M64 = 2 ** 64 - 1


def _mix(key: int, j: int) -> int:
    """splitmix64 of (key + (j + 1) * golden): the hash of the in-kernel replay sampler (csrc/learn.cu, dqn_mix)."""
    z = (key + (j + 1) * 0x9E3779B97F4A7C15) & _M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _M64
    return z ^ (z >> 31)


def q_net(state_dim: int, action_num: int, device, hidden=(64, 64)) -> torch.nn.Sequential:
    """A tanh MLP state_dim -> hidden... -> action_num with an identity head (torch's default init), the net shape
    K-DQN runs; used by the example and the tests."""
    dims = (int(state_dim), *[int(h) for h in hidden], int(action_num))
    layers = []
    for l in range(len(dims) - 1):
        layers.append(torch.nn.Linear(dims[l], dims[l + 1]))
        if l + 2 < len(dims):
            layers.append(torch.nn.Tanh())
    return torch.nn.Sequential(*layers).to(device)


class VecDQN(FlatAdam):
    def __init__(self, env, q_net: torch.nn.Module, dqn_msg: Optional[dict] = None, epsilon: float = 0.1, seed: int = 0,
                 group=None, track_episodes: bool = False):
        """The replay ring (``memory_capacity`` = R rows, all on the device):
        ``s [R, S, N]``, ``a [R, N]`` int32, ``r [R, N]``, ``s_ [R, S, N]`` float32, ``done [R, N]`` uint8,
        ``flag [R, N]`` int32.  Collection step k writes row k % R: the act kernel writes ``a``, the step kernel writes
        ``s_, r, done, flag`` and the policy-facing observation into ``s[(k + 1) % R]`` (no per-step copy).

        Invariant: that chained write replaces ``s`` of the oldest transition before its other fields are overwritten by
        the next step, so after k steps the ring samples only ``valid_rows = min(k, R - 1)`` rows, ending at
        ``newest_row = (k - 1) % R``; row ``k % R`` is in flight and never sampled.

        ``env``: a discrete-action env (``isActionContinuous is False``, one action dimension, ``action_space[0]`` the
        values of the ``action_num[0]`` indices) built with ``io_dtype=torch.float32, auto_reset=True``.  ``q_net``: tanh
        hidden layers and a linear head (e.g. :func:`q_net`) on ``env.device``: <= 4 layers, widths and state_dim <= 64,
        <= 64 actions.  Its parameters are moved into a flat buffer (the module keeps working).  ``epsilon``: the
        exploration probability of ``collect()``.  ``track_episodes``: per-episode statistics of every collected row in
        ``self.episodes``.  Single GPU: a process group of more than one rank raises ``ValueError``."""
        m = dict(DEFAULT_DQN_MSG)
        unknown = set(dqn_msg or {}) - set(m)
        if unknown:
            raise ValueError(f"VecDQN: unknown dqn_msg keys {sorted(unknown)}")
        m.update(dqn_msg or {})
        if getattr(env, 'isActionContinuous', True) is not False:
            raise ValueError("VecDQN needs a discrete-action env (isActionContinuous is False)")
        if env.action_dim != 1 or len(env.action_num) != 1:
            raise ValueError("VecDQN needs an env with one discrete action dimension")
        if env.io_dtype != torch.float32:
            raise ValueError("VecDQN: env must be built with io_dtype=torch.float32")
        if _dist.dist.is_available() and _dist.dist.is_initialized() and _dist.dist.get_world_size(group) > 1:
            raise ValueError("VecDQN runs on one GPU: the sampler's agreement over ranks is not designed yet")
        R, M = int(m['memory_capacity']), int(m['batch_size'])
        if R < 2 or M < 1 or int(m['target_replace_iter']) < 1 or int(m['learn_start']) < 1:
            raise ValueError("VecDQN: memory_capacity >= 2, batch_size, target_replace_iter and learn_start >= 1")
        if not math.isfinite(float(m['gamma'])):
            raise ValueError("VecDQN: gamma must be finite")
        self._check_epsilon(epsilon)
        layers = linear_layers(q_net)
        A = int(env.action_num[0])
        if not learn_fits(layers, 64):
            raise _lib.B200EnvError("K-DQN: the Q-net must have 1..4 linear layers with bias, widths and state_dim <= 64, "
                                    "<= 64 actions")
        if layers[0].in_features != env.state_dim or layers[-1].out_features != A:
            raise ValueError(f"VecDQN: the Q-net maps {layers[0].in_features} -> {layers[-1].out_features}, the env needs "
                             f"{env.state_dim} -> {A}")
        if getattr(env, 'host_only', False) or layers[0].weight.device.type != "cuda":
            raise _lib.B200EnvError("the engine has no CPU path: env and Q-net must live on a CUDA device")
        if not env.auto_reset:
            raise ValueError("VecDQN: env must be built with auto_reset=True")
        super().__init__([q_net], [m['lr']], m['betas'], m['adam_eps'], m['max_grad_norm'])
        self.env, self.q_net, self.msg, self.group = env, q_net, m, group
        self.R, self.batch_size, self.A = R, M, A
        self.gamma = float(m['gamma'])
        self.target_replace_iter, self.learn_start = int(m['target_replace_iter']), int(m['learn_start'])
        self.double_dqn = bool(m['double_dqn'])
        self.epsilon, self.seed = float(epsilon), int(seed)
        dev = env.device
        self.device = dev
        N, S = env.n_envs, env.state_dim
        f32 = dict(dtype=torch.float32, device=dev)
        self.s = torch.zeros((R, S, N), **f32)
        self.a = torch.zeros((R, N), dtype=torch.int32, device=dev)
        self.r = torch.zeros((R, N), **f32)
        self.s_ = torch.zeros((R, S, N), **f32)
        self.done = torch.zeros((R, N), dtype=torch.uint8, device=dev)
        self.flag = torch.zeros((R, N), dtype=torch.int32, device=dev)
        self.table = torch.tensor(env.action_space[0], **f32)    # the float32 image of action_space[0]
        self._value = torch.zeros((1, N), **f32)                  # the env's action buffer of a collection step

        self.target = self.params.flat.clone()
        self.q_mlp = self.params.mlp(0, 0)
        self.target_mlp = _lib.mlp(self.params.layers[0], 0, base=self.target)
        self.loss = torch.zeros(1, **f32)
        need = int(self._lib.b200_dqn_workspace_bytes(C.byref(self.q_mlp), M))
        if need == 0:
            raise _lib.B200EnvError("b200_dqn_workspace_bytes: net not supported by K-DQN")
        self.workspace = torch.zeros(need, dtype=torch.uint8, device=dev)
        self._key0 = (self.seed * 0x9E3779B97F4A7C15 + 0x44514E5253) & _M64

        self.episodes = EpisodeTracker(N, dev) if track_episodes else None
        self.k = 0                 # collection steps so far (the Philox step of the next one)
        self.updates = 0           # learn() updates so far
        self._started = False

    # ------------------------------------------------------------------ small pieces
    @staticmethod
    def _check_epsilon(eps) -> None:
        if not (0.0 <= float(eps) <= 1.0):
            raise ValueError("epsilon must lie in [0, 1]")

    def set_epsilon(self, epsilon: float) -> None:
        self._check_epsilon(epsilon)
        self.epsilon = float(epsilon)

    @property
    def valid_rows(self) -> int:
        return min(self.k, self.R - 1)

    @property
    def newest_row(self) -> int:
        return (self.k - 1) % self.R

    def sample_key(self, update: int) -> int:
        """The sampling key of update number ``update`` (0-based): a hash of ``seed`` and the update counter."""
        return _mix(self._key0, int(update))

    def act(self, obs_soa: torch.Tensor, index: torch.Tensor, value: torch.Tensor, epsilon: float, step: int,
            q: Optional[torch.Tensor] = None) -> None:
        """``b200_dqn_act`` on ``obs_soa [S, N]`` -> ``index [N]`` int32, ``value [1, N]`` (and ``q [A, N]``)."""
        N = obs_soa.shape[1]
        p = _lib.ptr
        with torch.cuda.device(self.device):
            _lib.check(self._lib.b200_dqn_act(
                N, C.byref(self.q_mlp), p(obs_soa), p(self.table), float(epsilon), self.seed & _M64, int(step) & _M64,
                self.env.env_index_offset, p(index), p(value), p(q), self._stream()), "b200_dqn_act")

    # ------------------------------------------------------------------ collection
    def collect(self, steps: int) -> None:
        """``steps`` epsilon-greedy steps of all N instances into the ring (no host copy, no synchronisation)."""
        env, R = self.env, self.R
        if not self._started:
            env.reset(True)
            if self.episodes is not None:
                self.episodes.reset_carry()
            self.s[self.k % R].copy_(env._reset_obs)
            self._started = True
        left = int(steps)
        while left > 0:
            row0 = self.k % R
            seg = min(left, R - row0)          # a contiguous run of rows: the episode scan reads it before it wraps
            for t in range(row0, row0 + seg):
                self.act(self.s[t], self.a[t], self._value, self.epsilon, self.k)
                env.step_into(self._value, obs=None, next_obs=self.s_[t], reward=self.r[t], done=self.done[t],
                              flag=self.flag[t], policy_obs=self.s[(t + 1) % R])
                self.k += 1
            if self.episodes is not None:
                sl = slice(row0, row0 + seg)
                self.episodes.update(self.r[sl], self.done[sl], self.flag[sl])
            left -= seg

    # ------------------------------------------------------------------ update
    def _batch(self, sample_key: int, index: Optional[torch.Tensor]) -> _lib.DQNBatch:
        b = _lib.DQNBatch()
        b.R, b.N = self.R, self.env.n_envs
        b.s, b.r, b.s_, b.a, b.done = (t.data_ptr() for t in (self.s, self.r, self.s_, self.a, self.done))
        b.newest_row, b.valid_rows = self.newest_row, self.valid_rows
        b.count = self.batch_size if index is None else index.numel()
        b.index = None if index is None else index.data_ptr()
        b.sample_key = int(sample_key) & _M64
        return b

    def grad_step(self, sample_key: int, index: Optional[torch.Tensor] = None) -> None:
        """The gradient of one mini-batch (``b200_dqn_grad``) -> ``self.grad``, ``self.loss``.  ``index``: device int64
        ring positions (row * N + i) instead of the keyed draw."""
        if index is not None and not (index.is_cuda and index.dtype == torch.int64 and index.is_contiguous()):
            raise ValueError("grad_step: index must be a contiguous CUDA int64 tensor")
        b = self._batch(sample_key, index)
        p = _lib.ptr
        with torch.cuda.device(self.device):
            _lib.check(self._lib.b200_dqn_grad(
                C.byref(b), C.byref(self.q_mlp), C.byref(self.target_mlp), self.gamma, int(self.double_dqn), p(self.grad),
                p(self.loss), p(self.workspace), self.workspace.numel(), self._stream()), "b200_dqn_grad")

    def learn(self, updates: int = 1) -> Optional[dict]:
        """``updates`` x (target copy when due, gradient, Adam).  Returns None (and does nothing) while fewer than
        ``learn_start`` ring rows are valid; else ``{"loss": loss of the last update}`` (one host read)."""
        if self.valid_rows < self.learn_start:
            return None
        for _ in range(int(updates)):
            if self.updates % self.target_replace_iter == 0:
                self.target.copy_(self.params.flat)
            self.grad_step(self.sample_key(self.updates))
            self.adam_step()
            self.updates += 1
        return {"loss": float(self.loss)}

    # ------------------------------------------------------------------ evaluation
    def evaluate(self, obs_soa: torch.Tensor):
        """Greedy action of ``[state_dim, N]`` observations: ``(index [N] int32, value [1, N] float32)``."""
        N = obs_soa.shape[1]
        index = torch.empty(N, dtype=torch.int32, device=self.device)
        value = torch.empty(1, N, dtype=torch.float32, device=self.device)
        self.act(obs_soa.contiguous(), index, value, 0.0, 0)
        return index, value

    def evaluate_episodes(self, env, max_steps: int) -> dict:
        """The greedy policy (epsilon = 0) on every instance of ``env`` for one whole episode each, as
        :meth:`VecPPO2.evaluate_episodes`: ``env`` is a separate instance of the training env's class (``auto_reset``,
        float32 io), reset here and stepped until every instance has finished an episode (checked every 64 steps) or
        ``max_steps`` steps have run.  Nothing of the agent changes.  Returns ``ep_return``, ``ep_length``, ``ep_flag``
        ([N] device tensors; NaN / -1 = unfinished) and the keys of :meth:`EpisodeTracker.summary`."""
        if env.state_dim != self.env.state_dim:
            raise ValueError("evaluate_episodes: env dimensions differ from the Q-net's")
        index = torch.empty(env.n_envs, dtype=torch.int32, device=env.device)
        value = torch.empty(1, env.n_envs, dtype=torch.float32, device=env.device)
        act = lambda obs: self.act(obs, index, value, 0.0, 0)
        return evaluate_first_episodes(self.env, env, act, value, max_steps, self.group)
