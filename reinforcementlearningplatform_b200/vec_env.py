"""Vector mirror of the reference env contract ``algorithm/rl_base.py:4-162``.

The reference exposes one instance per Python object; its ``train.py`` loops
read ``state_dim / action_dim / action_range / name / dt / timeMax|time_max``
and, every step, ``current_state, next_state, reward, is_terminal,
terminal_flag, time`` after calling ``step_update(action)`` (e.g.
``demonstration/PPO2/PPO2-4-CartPoleAngleOnly/train.py:138-215``).

``VecEnvBase`` keeps exactly those names but with a leading instance axis
(torch CUDA tensors, owned by the env and overwritten in place each step --
``.clone()`` replaces the reference's ``.copy()``).  All arithmetic happens in
``libb200env.so`` (hand-written sm_100a kernels); this file only owns buffers
and fills the parameter struct from the reference attribute names.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import math

import numpy as np
import torch

from . import _lib


class VecEnvBase:
    ENV_ID: int = -1
    VARIANT: int = 0
    STATE_FIELDS: tuple = ()  # names of the SoA state fields, in storage order
    # True where get_state() is a pure function of the persistent state, so that the pre-step `current_state` of step
    # t+1 is bit-identical to the policy-facing observation written by step t (s' or the reset observation).  Such envs
    # do not recompute it: the two buffers swap roles and the kernel is launched with io.obs = NULL (for the fake laser
    # of UGVForwardObstacleAvoidance this removes one of the two 37-ray scans per step, SURVEY 8d).  Not true for the
    # UAV envs (the reset observation is taken against the stale reference) nor the two-link arm (pre-wrap error).
    OBS_IS_PURE: bool = False
    TIMEOUT_FLAG: int = 0  # terminal_flag value of a time-out (train loops: success = done and flag != TIMEOUT_FLAG)
    USES_WORK_LIST: bool = False  # the step kernel wants b200env_io.work (list of terminated instances)

    def __init__(self, n_envs: int = 1, device="cuda", dtype=torch.float64, seed: int = 0,
                 env_index_offset: int = 0, auto_reset: bool = False, host_only: bool = False, io_dtype=None,
                 reuse_obs: Optional[bool] = None):
        """``dtype``: type of the persistent state and of all arithmetic.  ``io_dtype``: type of the RL-facing buffers
        (action, dis, current/next/policy state, reward); default = ``dtype``.  ``dtype=float64, io_dtype=float32`` keeps
        the reference's fp64 trajectories while exchanging float32 with the (float32) policy and rollout buffer, as the
        reference does at ``RolloutBuffer.to_tensor`` (utils/classes.py:292-301)."""
        if dtype not in (torch.float64, torch.float32):
            raise ValueError("dtype must be torch.float64 or torch.float32")
        io_dtype = dtype if io_dtype is None else io_dtype
        if io_dtype not in (dtype, torch.float32):
            raise ValueError("io_dtype must equal dtype or be torch.float32")
        self.io_dtype = io_dtype
        self._params = self.make_params()
        self.host_only = bool(host_only)
        if host_only:  # parameter/attribute mirror only (CPU tests, oracle drivers): no buffers, no launches
            self.n_envs, self.dtype = int(n_envs), dtype
            try:  # b200env_dims is a host function of the library; without a built library the mirror has no dims
                _, self.state_dim, self.action_dim, _ = _lib.dims(self.ENV_ID, self.VARIANT)
            except (OSError, _lib.B200EnvError):
                pass
            return
        self._lib = _lib.load()  # raises if the CUDA engine is not built
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.B200EnvError("the engine has no CPU path: device must be a CUDA device")
        self.n_envs = int(n_envs)
        self.dtype = dtype
        self._dt_code = _lib.F64 if dtype == torch.float64 else _lib.F32
        self.seed = int(seed)
        self.env_index_offset = int(env_index_offset)
        self.auto_reset = bool(auto_reset)
        self.reuse_obs = self.OBS_IS_PURE if reuse_obs is None else (bool(reuse_obs) and self.OBS_IS_PURE)
        self._policy_obs_valid = False  # _reset_obs holds get_state() of the current persistent state for every lane
        self._hot_io = None             # cached b200env_io of step_soa

        sf, od, ad, dd = _lib.dims(self.ENV_ID, self.VARIANT)
        assert sf == len(self.STATE_FIELDS), (sf, self.STATE_FIELDS)
        self._sf, self._od, self._ad, self._dd = sf, od, ad, dd
        N, dev = self.n_envs, self.device
        z = lambda *shape, dt=io_dtype: torch.zeros(*shape, dtype=dt, device=dev)
        # the buffer the kernels see: field-major [sf, N], or block-interleaved [blocks, slots, B] (UAV families,
        # include/b200env.h b200env_state_layout); `self._state` is always the logical [sf, N] picture
        self._blk, self._slots = _lib.state_layout(self.ENV_ID, self.VARIANT)
        if self._blk:
            self._state_raw = z((N + self._blk - 1) // self._blk, self._slots, self._blk, dt=dtype)
        else:
            self._state_raw = z(sf, N, dt=dtype)
        self._time = z(N, dt=torch.float64)
        self._episode = z(N, dt=torch.int32)  # bit pattern of the u32 episode counter
        self._obs = z(od, N)
        self._next_obs = z(od, N)
        self._reset_obs = z(od, N)
        self._reward = z(N)
        self._done = z(N, dt=torch.uint8)
        self._flag = z(N, dt=torch.int32)
        self._action = z(ad, N)
        self._work = z(N + 1, dt=torch.int32) if self.USES_WORK_LIST else None  # b200env_io.work

        '''rl_base'''
        self.state_dim = od
        self.action_dim = ad
        self.current_action = self._action.t()
        self.is_terminal = self._done.view(torch.bool)
        self.terminal_flag = self._flag
        self.reward = self._reward
        self.time = self._time
        '''rl_base'''

    # ------------------------------------------------------------------ params
    def make_params(self) -> C.Structure:
        raise NotImplementedError

    # ------------------------------------------------------------------ rl_base metadata (algorithm/rl_base.py:5-124)
    # Descriptive lists the reference keeps next to state_dim / action_dim; the info printers and the PPO / DQN scripts read
    # them.  Every env of the engine is continuous in state and action unless a subclass says otherwise
    # (FlightAttitudeSimulatorDiscrete defines action_num / action_space itself).
    _RL_BASE_LISTS = {"state_num": ("state_dim", math.inf), "state_step": ("state_dim", None), "state_space": ("state_dim", None),
                      "isStateContinuous": ("state_dim", True), "state_range": ("state_dim", (-math.inf, math.inf)),
                      "action_num": ("action_dim", math.inf), "action_step": ("action_dim", None),
                      "action_space": ("action_dim", None), "isActionContinuous": ("action_dim", True)}

    def __getattr__(self, name):  # only reached for names that are not set on the instance or its class
        spec = VecEnvBase._RL_BASE_LISTS.get(name)
        if spec is not None:
            dim = getattr(self, spec[0])
            return [list(spec[1]) if isinstance(spec[1], tuple) else spec[1] for _ in range(int(dim))]
        raise AttributeError(f"{type(self).__name__!s} has no attribute {name!r}")

    @property
    def current_state_norm(self):
        """``Normalization(state_dim)`` applied by the train loops to ``current_state`` (uav_pos_ctrl_RL.py:36,
        SecondOrderIntegration.py:76, PPO2-4-UavFntsmcParamPos/train.py:291); device-resident, see normalization.py."""
        if getattr(self, "_cur_norm", None) is None:
            from .normalization import Normalization
            self._cur_norm = Normalization(self.state_dim, device=self.device)
        return self._cur_norm

    @property
    def next_state_norm(self):
        if getattr(self, "_next_norm", None) is None:
            from .normalization import Normalization
            self._next_norm = Normalization(self.state_dim, device=self.device)
        return self._next_norm

    _NORM_COLS = ("cur_n", "cur_mean", "cur_std", "cur_S", "next_n", "next_mean", "next_std", "next_S")

    def save_state_norm(self, path, msg=None):
        """Same CSV as uav_pos_ctrl_RL.py:208-222 / SecondOrderIntegration.py:354-368 (columns cur_n, cur_mean, cur_std, cur_S,
        next_n, ...); the PPO2 train scripts of every env call it."""
        c, x = self.current_state_norm.running_ms, self.next_state_norm.running_ms
        cols = [c.n * np.ones(self.state_dim), c.mean, c.std, c.S, x.n * np.ones(self.state_dim), x.mean, x.std, x.S]
        name = path + ('state_norm.csv' if msg is None else 'state_norm_' + msg + '.csv')
        np.savetxt(name, np.stack(cols, axis=1), delimiter=',', header=','.join(self._NORM_COLS), comments='', fmt='%.17g')

    def load_norm_normalizer_from_file(self, path, file):
        """uav_pos_ctrl_RL.py:224-233; reads the reference's own ``state_norm.csv`` files."""
        data = np.atleast_2d(np.genfromtxt(path + file, delimiter=',', skip_header=1))
        c, x = self.current_state_norm.running_ms, self.next_state_norm.running_ms
        c.n, c.mean, c.S = data[0, 0], data[:, 1], data[:, 3]
        x.n, x.mean, x.S = data[0, 4], data[:, 5], data[:, 7]


    def _io(self, action=None, dis=None, obs=True, reset_obs=True) -> _lib.IO:
        io = _lib.IO()
        io.state = self._state_raw.data_ptr()
        io.time = self._time.data_ptr()
        io.episode = self._episode.data_ptr()
        io.action = None if action is None else action.data_ptr()
        io.dis = None if dis is None else dis.data_ptr()
        io.obs = self._obs.data_ptr() if obs else None
        io.next_obs = self._next_obs.data_ptr()
        io.reward = self._reward.data_ptr()
        io.done = self._done.data_ptr()
        io.flag = self._flag.data_ptr()
        io.reset_obs = self._reset_obs.data_ptr() if reset_obs else None
        io.work = None if self._work is None else self._work.data_ptr()
        io.io_dtype = _lib.F32 if (self.io_dtype == torch.float32 and self.dtype == torch.float64) else _lib.F64
        return io

    def _as_soa(self, x, rows: int, layout: Optional[str] = None) -> torch.Tensor:
        """Accept [N, rows] (reference orientation) or [rows, N] (engine SoA).  A 1-D vector of ``rows`` values is one
        action broadcast to every instance; of ``N`` values (rows == 1) one value per instance.  When n_envs == rows a
        2-D input fits both orientations: ``layout`` ("rows_first" = [rows, N] or "envs_first" = [N, rows]) must then
        say which one is meant -- guessing would silently hand every instance the wrong action components."""
        if not torch.is_tensor(x):
            x = torch.as_tensor(np.asarray(x), dtype=self.io_dtype)
        x = x.to(device=self.device, dtype=self.io_dtype)
        if x.dim() == 1:
            if rows == 1 and x.numel() == self.n_envs:
                return x.view(1, -1).contiguous()
            if x.numel() != rows:
                raise ValueError(f"expected {rows} values (one action for all instances), got {x.numel()}")
            return x.view(-1, 1).expand(rows, self.n_envs).contiguous()
        if layout not in (None, "rows_first", "envs_first"):
            raise ValueError("layout must be 'rows_first' or 'envs_first'")
        ef, rf = x.shape == (self.n_envs, rows), x.shape == (rows, self.n_envs)
        if ef and rf and layout is None and rows > 1:
            raise ValueError(f"a [{rows},{rows}] input is ambiguous when n_envs == {rows}: pass layout='envs_first' "
                             "([N, dim], the reference's orientation) or layout='rows_first' ([dim, N], engine SoA)")
        if ef and layout != "rows_first":
            return x.t().contiguous()
        if rf and layout != "envs_first":
            return x.contiguous()
        raise ValueError(f"expected [{self.n_envs},{rows}] or [{rows},{self.n_envs}], got {tuple(x.shape)}")

    # ------------------------------------------------------------- rl_base API
    @property
    def current_state(self) -> torch.Tensor:
        """[N, state_dim] view of the pre-step observation (rl_base.py:22)."""
        return self._obs.t()

    @property
    def next_state(self) -> torch.Tensor:
        """[N, state_dim] view of s' (rl_base.py:23)."""
        return self._next_obs.t()

    @property
    def policy_state(self) -> torch.Tensor:
        """[N, state_dim] observation to act on next: s' or the reset observation after an auto-reset."""
        return self._reset_obs.t()

    def reset(self, random: bool = True, mask: Optional[torch.Tensor] = None) -> None:
        """``env.reset(random)`` (rl_base.py:161) for all instances or those in ``mask``."""
        if random:
            with torch.cuda.device(self.device):
                io = self._io(obs=False, reset_obs=False)
                m = None
                if mask is not None:
                    m = mask.to(device=self.device, dtype=torch.uint8).contiguous()
                _lib.check(self._lib.b200env_reset(self.ENV_ID, self._dt_code, self.n_envs, C.byref(self._params),
                                                   C.sizeof(self._params), C.byref(io), _lib.ptr(m), self.seed,
                                                   self.env_index_offset, _lib.stream(self.device)), "b200env_reset")
        else:
            self._reset_default(mask)
            if mask is None:
                self.observe()
            else:  # get_state() of the re-initialised lanes only: the other lanes keep their next_state (s' of the last step)
                keep = self._next_obs.clone()
                self.observe()
                m = mask.to(self.device).bool()
                self._next_obs[:, ~m] = keep[:, ~m]
        sel = slice(None) if mask is None else mask.to(self.device).bool()
        self._obs[:, sel] = self._next_obs[:, sel]
        self._reset_obs[:, sel] = self._next_obs[:, sel]
        self._reward[sel] = 0
        self._done[sel] = 0
        self._flag[sel] = 0
        if mask is None:
            self._policy_obs_valid = True

    def _reset_default(self, mask) -> None:
        raise NotImplementedError

    def observe(self) -> torch.Tensor:
        """``env.get_state()`` (rl_base.py:158) of the current state, into ``next_state``."""
        with torch.cuda.device(self.device):
            io = self._io(obs=False, reset_obs=False)
            _lib.check(self._lib.b200env_observe(self.ENV_ID, self._dt_code, self.n_envs, C.byref(self._params),
                                                 C.sizeof(self._params), C.byref(io), _lib.stream(self.device)),
                       "b200env_observe")
        return self.next_state

    get_state = observe

    def step_update(self, action, dis=None, layout: Optional[str] = None) -> None:
        """``env.step_update(action)`` (rl_base.py:126) for every instance; results land in
        ``current_state, next_state, reward, is_terminal, terminal_flag`` like the reference.  ``layout``: see
        :meth:`_as_soa` (only needed when n_envs == action_dim)."""
        a = self._as_soa(action, self._ad, layout)
        self._action = a
        self.current_action = a.t()
        d = None if dis is None else self._as_soa(dis, self._dd, layout)
        self.step_soa(a, d)

    def step_soa(self, action_soa: torch.Tensor, dis_soa: Optional[torch.Tensor] = None) -> None:
        """Hot call: ``action_soa`` is ``[action_dim, N]`` contiguous in ``io_dtype`` (no copies made).  The host side of
        a step is ~6 us of Python: the I/O struct is cached and only the pointers that change are rewritten."""
        if action_soa.dtype != self.io_dtype or (dis_soa is not None and dis_soa.dtype != self.io_dtype):
            raise _lib.B200EnvError(f"step_soa: action/dis must be {self.io_dtype}")
        reuse = self.reuse_obs and self._policy_obs_valid
        if reuse:  # current_state(t+1) == policy_state(t): swap the buffers instead of recomputing get_state()
            self._obs, self._reset_obs = self._reset_obs, self._obs
        io = self._hot_io
        if io is None:
            io = self._hot_io = self._io()
            self._hot_args = (self.ENV_ID, self._dt_code, self.n_envs, C.byref(self._params), C.sizeof(self._params),
                              C.byref(io))
            self._dev_index = self._state_raw.device.index
        io.action = action_soa.data_ptr()
        io.dis = None if dis_soa is None else dis_soa.data_ptr()
        io.obs = None if reuse else self._obs.data_ptr()
        io.reset_obs = self._reset_obs.data_ptr()
        self._policy_obs_valid = True
        stream = torch.cuda.current_stream(self._state_raw.device).cuda_stream
        if torch.cuda.current_device() != self._dev_index:
            with torch.cuda.device(self._dev_index):
                rc = self._lib.b200env_step(*self._hot_args, _lib.AUTO_RESET if self.auto_reset else 0, self.seed,
                                            self.env_index_offset, stream)
        else:
            rc = self._lib.b200env_step(*self._hot_args, _lib.AUTO_RESET if self.auto_reset else 0, self.seed,
                                        self.env_index_offset, stream)
        if rc:
            _lib.check(rc, "b200env_step")

    def step_into(self, action_soa: torch.Tensor, dis_soa: Optional[torch.Tensor] = None, *, obs: Optional[torch.Tensor],
                  next_obs: torch.Tensor, reward: torch.Tensor, done: torch.Tensor, flag: torch.Tensor,
                  policy_obs: Optional[torch.Tensor] = None) -> None:
        """``step_soa`` with the outputs of this step stored into caller-owned tensors (one row of a device-resident
        ``rollout.RolloutBuffer``) instead of the env's own ``current_state / next_state / reward / is_terminal /
        terminal_flag`` buffers, which are left untouched.  Shapes: ``obs, next_obs [state_dim, N]``, ``reward [N]`` in
        ``io_dtype``; ``done [N]`` uint8; ``flag [N]`` int32.  ``obs=None``: ``current_state`` is not stored (the kernels
        skip it).  ``policy_obs``: where the observation the policy acts on next (``next_state``, or the reset observation
        after an auto-reset) is written instead of ``env.policy_state`` -- a collection loop passes the NEXT row of its
        observation buffer, so that the row is in place when the policy reads it and no copy is made; the caller then owns
        that chain (``env.policy_state`` is stale until a step writes it again)."""
        io_dt = self.io_dtype
        checks = [(next_obs, (self._od, self.n_envs), io_dt), (reward, (self.n_envs,), io_dt),
                  (done, (self.n_envs,), torch.uint8), (flag, (self.n_envs,), torch.int32)]
        if obs is not None:
            checks.append((obs, (self._od, self.n_envs), io_dt))
        if policy_obs is not None:
            checks.append((policy_obs, (self._od, self.n_envs), io_dt))
        for t, shape, dt in checks:
            if tuple(t.shape) != shape or t.dtype != dt or not t.is_contiguous() or t.device != self._state_raw.device:
                raise _lib.B200EnvError(f"step_into: expected contiguous {dt} tensor of shape {shape} on {self.device}")
        if action_soa.dtype != io_dt or (dis_soa is not None and dis_soa.dtype != io_dt):
            raise _lib.B200EnvError(f"step_into: action/dis must be {io_dt}")
        with torch.cuda.device(self.device):
            reuse = self.reuse_obs and self._policy_obs_valid
            if reuse and obs is not None:  # current_state(t) == policy_state(t-1): a row copy instead of a second get_state()
                obs.copy_(self._reset_obs)
            io = self._io(action_soa, dis_soa, obs=False)
            if not reuse and obs is not None:
                io.obs = obs.data_ptr()
            io.next_obs, io.reward, io.done, io.flag = next_obs.data_ptr(), reward.data_ptr(), done.data_ptr(), flag.data_ptr()
            if policy_obs is not None:
                io.reset_obs = policy_obs.data_ptr()
            self._policy_obs_valid = policy_obs is None or policy_obs.data_ptr() == self._reset_obs.data_ptr()
            flags = _lib.AUTO_RESET if self.auto_reset else 0
            _lib.check(self._lib.b200env_step(self.ENV_ID, self._dt_code, self.n_envs, C.byref(self._params),
                                              C.sizeof(self._params), C.byref(io), flags, self.seed,
                                              self.env_index_offset, _lib.stream(self.device)), "b200env_step")

    def rollout_into(self, steps: int, action: torch.Tensor, *, obs: torch.Tensor, next_obs: torch.Tensor,
                     reward: torch.Tensor, done: torch.Tensor, flag: torch.Tensor,
                     dis: Optional[torch.Tensor] = None) -> None:
        """``steps`` control periods with pre-computed actions in ONE call (``b200env_rollout``): time-major tensors
        ``action [steps, action_dim, N]``, ``obs / next_obs [steps, state_dim, N]``, ``reward [steps, N]`` in ``io_dtype``,
        ``done [steps, N]`` uint8, ``flag [steps, N]`` int32 (rows of a ``rollout.RolloutBuffer``).  The FAS / SOI /
        BallBalancer / TwoLink / UGV families run all steps in one kernel with the state in registers."""
        T, N = int(steps), self.n_envs
        chk = ((action, (T, self._ad, N), self.io_dtype), (obs, (T, self._od, N), self.io_dtype),
               (next_obs, (T, self._od, N), self.io_dtype), (reward, (T, N), self.io_dtype),
               (done, (T, N), torch.uint8), (flag, (T, N), torch.int32))
        for t, shape, dt in chk:
            if tuple(t.shape) != shape or t.dtype != dt or not t.is_contiguous() or t.device != self._state_raw.device:
                raise _lib.B200EnvError(f"rollout_into: expected contiguous {dt} tensor of shape {shape}")
        if dis is not None and (tuple(dis.shape) != (T, self._dd, N) or dis.dtype != self.io_dtype or not dis.is_contiguous()):
            raise _lib.B200EnvError("rollout_into: bad dis tensor")
        spec = _lib.RolloutSpec(T, self._ad * N, self._dd * N, self._od * N, self._od * N, N, N, N)
        with torch.cuda.device(self._state_raw.device):
            io = self._io(action, dis)
            io.obs, io.next_obs, io.reward = obs.data_ptr(), next_obs.data_ptr(), reward.data_ptr()
            io.done, io.flag = done.data_ptr(), flag.data_ptr()
            _lib.check(self._lib.b200env_rollout(self.ENV_ID, self._dt_code, N, C.byref(self._params),
                                                 C.sizeof(self._params), C.byref(io), C.byref(spec),
                                                 _lib.AUTO_RESET if self.auto_reset else 0, self.seed,
                                                 self.env_index_offset, _lib.stream(self.device)), "b200env_rollout")
        self._policy_obs_valid = True

    def get_reward(self) -> torch.Tensor:
        return self._reward

    def is_Terminal(self) -> torch.Tensor:
        return self.is_terminal

    # ------------------------------------------------------- logical view of the persistent state
    @property
    def _state(self) -> torch.Tensor:
        """The persistent state as ``[state_fields, N]``.  Field-major envs: the device buffer itself (writes go through).
        Block-interleaved envs (UAV): a COPY in logical order -- write back with ``_write_state``."""
        if not self._blk:
            return self._state_raw
        raw = self._state_raw
        nb, slots, B = raw.shape
        return raw.permute(1, 0, 2).reshape(slots, nb * B)[:self._sf, :self.n_envs].contiguous()

    def _write_state(self, logical: torch.Tensor) -> None:
        """Logical ``[state_fields, N]`` -> the device layout."""
        logical = torch.as_tensor(logical).to(self.device, self.dtype)
        if not self._blk:
            self._state_raw.copy_(logical)
            return
        raw = self._state_raw
        nb, slots, B = raw.shape
        full = torch.zeros(slots, nb * B, dtype=self.dtype, device=self.device)
        full[:self._sf, :self.n_envs] = logical
        raw.copy_(full.view(slots, nb, B).permute(1, 0, 2))

    # ------------------------------------------------------- state injection
    def get_state_buffers(self) -> dict:
        return {"state": self._state.clone(), "time": self._time.clone(), "episode": self._episode.clone()}

    def set_state_buffers(self, state=None, time=None, episode=None) -> None:
        """Inject SoA state ([fields, N]), time ([N]) -- parity re-sync and checkpoint restore."""
        self._policy_obs_valid = False  # the next step recomputes current_state in-kernel
        if state is not None:
            self._write_state(state)
        if time is not None:
            self._time.copy_(torch.as_tensor(time).to(self.device, torch.float64))
        if episode is not None:
            self._episode.copy_(torch.as_tensor(episode).to(self.device, torch.int32))

    def field(self, name: str) -> torch.Tensor:
        return self._state[self.STATE_FIELDS.index(name)]
