"""GPU: the small-env kernels on the edge lanes of tests/env_edges.py -- every terminal threshold, clamp, wrap, time-out
and sub-step count within a few ulps.

  parked / time lanes   flag, done, reward and post-step time equal the C oracle's bit for bit, the rest within
                        ENGINE_TOL; auto-resets take the oracle's Philox draws.
  crossing lanes        the engine's flag (and reward branch) equal the reference rule applied to the engine's OWN
                        post-step state, in every lane; the state is within ENGINE_TOL of the oracle's.
  float32 I/O           decides exactly like fp64; every RL-facing output is the fp64 value rounded once.
  fp32                  parked and time lanes follow the float32 restatement of each rule (thresholds `(T)p.x`, time
                        in float64); parked states keep their bits.
  rollout               the fused multi-step kernel (b200env_rollout) writes the bits of the same steps launched one by
                        one.
"""
import numpy as np
import pytest

import env_edges as E
from helpers import ENGINE_TOL, env_specs

pytestmark = pytest.mark.gpu


def _env(name, n, dtype, io_dtype=None, auto_reset=False):
    cls, kw = env_specs()[name]
    return cls(n_envs=n, device="cuda", dtype=dtype, io_dtype=io_dtype, seed=E.SEED, auto_reset=auto_reset, **kw)


def _inject(env, L):
    import torch
    env.set_state_buffers(torch.from_numpy(np.ascontiguousarray(L.state.T)), torch.from_numpy(L.time),
                          torch.zeros(len(L.time), dtype=torch.int32))


def engine_step(name, L, dtype=None, io_dtype=None, auto_reset=False):
    """one step launch on the lanes -> lanes-first float64 outputs (and the raw io-dtype ones under 'raw_*')."""
    import torch
    dtype = dtype or torch.float64
    env = _env(name, len(L.time), dtype, io_dtype, auto_reset)
    _inject(env, L)
    a = torch.from_numpy(np.ascontiguousarray(L.action.T)).to("cuda", env.io_dtype)
    env.step_soa(a)
    torch.cuda.synchronize()
    f = lambda x: x.detach().cpu().numpy()
    out = dict(obs=f(env._obs).T, next_obs=f(env._next_obs).T, reset_obs=f(env._reset_obs).T, reward=f(env._reward),
               done=f(env._done), flag=f(env._flag), state=f(env._state).T, time=f(env._time),
               episode=f(env._episode).view(np.uint32))
    return {k: (v.astype(np.float64) if v.dtype.kind == "f" else v) for k, v in out.items()} | {
        "raw_" + k: out[k] for k in ("obs", "next_obs", "reset_obs", "reward", "state")}


def _mixed(a, b):
    return np.max(np.abs(a - b) / np.maximum(1.0, np.abs(b)), axis=tuple(range(1, a.ndim))) if a.ndim > 1 else \
        np.abs(a - b) / np.maximum(1.0, np.abs(b))


def _where(L, m, limit=8):
    idx = np.nonzero(m)[0][:limit]
    return [(str(L.label[i]), int(L.k[i]), int(i)) for i in idx]


def _sel(L, mask):
    return E.Lanes(L.state[mask], L.time[mask], L.action[mask], L.label[mask], L.kind[mask], L.k[mask])


@pytest.mark.parametrize("name", E.NAMES)
def test_parked_and_time_lanes_equal_the_oracle(name, oracle_lib):
    L = E.lanes(name)
    L = _sel(L, np.isin(L.kind, ["parked", "priority", "time"]))
    g = engine_step(name, L, auto_reset=True)
    o = E.oracle_step(name, L.state, L.time, L.action, auto_reset=True)
    tol = ENGINE_TOL[name]
    for k in ("flag", "done", "time", "episode"):
        bad = g[k] != o[k]
        assert not bad.any(), (name, k, int(bad.sum()), _where(L, bad))
    # the reward has the oracle's bits wherever the state did not move (so the engine's equals the oracle's) and the
    # reward holds no transcendental: UGV's heading term -|ephi| Q_phi (atan2, taken when e > 0.1) is within ENGINE_TOL
    still = E.oracle_step(name, L.state, L.time, L.action)["state"]   # before any auto-reset
    exact = np.all(still == L.state, axis=1)
    if name in E.UGV_NAMES or name == "ugvo":   # (UGV-FOA's demo-copy reward has no heading term)
        tx, ty = (L.state[:, 5], L.state[:, 6]) if name == "ugvo" else (E.host(name)._params.target_x, E.host(name)._params.target_y)
        exact &= E.np_norm2(tx - L.state[:, 0], ty - L.state[:, 1]) <= 0.1
    bad = np.where(exact, g["reward"] != o["reward"], _mixed(g["reward"], o["reward"]) > tol)
    assert not bad.any(), (name, "reward", int(bad.sum()), _where(L, bad))
    assert exact.sum() > 0 or name in ("cartpole_angleonly_ppo2", "fas", "fas_ppo2", "fas_discrete"), name
    for k in ("state", "next_obs", "reset_obs", "obs"):
        bad = _mixed(g[k], o[k]) > tol
        assert not bad.any(), (name, k, int(bad.sum()), _where(L, bad))


@pytest.mark.parametrize("name", E.NAMES)
def test_crossing_lanes_follow_the_reference_rule(name, oracle_lib):
    """the flag of every lane equals the reference rule evaluated on the engine's own post-step state (exact: the decisive
    values are all outputs), the other decisions too; states within ENGINE_TOL of the oracle's."""
    L = E.lanes(name)
    p = E.host(name)._params
    g = engine_step(name, L)
    o = E.oracle_step(name, L.state, L.time, L.action)
    want = E.rule_flag(name, p, L.state, g["state"], g["time"])
    bad = g["flag"] != want
    per = {lab: int(n) for lab, n in zip(*np.unique(L.label[bad], return_counts=True))} if bad.any() else {}
    assert not bad.any(), (name, f"{int(bad.sum())} of {len(bad)} lanes decide against the rule", per, _where(L, bad))
    assert np.array_equal(g["done"], (g["flag"] != 0).astype(np.uint8))
    for what, m in E.rule_extras(name, p, g).items():
        assert not m.any(), (name, what, int(m.sum()), _where(L, m))
    assert np.array_equal(g["time"], o["time"]), name
    tol = ENGINE_TOL[name]
    err = E.state_compare(name, p, g["state"], o["state"])
    if name == "fas_discrete":
        # the -0.8 bounce makes dtheta jump where the two sides clamp differently; that happens only where the pre-clamp
        # angles straddle theta_max, i.e. both post-step angles are on it within an ulp or two
        ce, co = np.abs(g["state"][:, 0]) == p.theta_max, np.abs(o["state"][:, 0]) == p.theta_max
        split = ce != co
        assert np.all(np.abs(np.abs(g["state"][split, 0]) - p.theta_max) <= 4e-16), name
        err = np.where(split, 0.0, err)
    bad = err > tol
    assert not bad.any(), (name, "state", int(bad.sum()), float(err.max()), _where(L, bad))
    # lanes where both sides took the same branches (flag, wrap, clamp, reward) have comparable outputs
    same = (g["flag"] == o["flag"]) & (_mixed(g["state"], o["state"]) <= tol)
    bg, bo = E.reward_branch(name, p, g), E.reward_branch(name, p, o)
    if bg is not None:
        same &= bg == bo
    for k in ("next_obs", "reward"):
        e = _mixed(g[k], o[k])
        bad = same & (e > tol)
        assert not bad.any(), (name, k, int(bad.sum()), _where(L, bad))


@pytest.mark.parametrize("name", E.NAMES)
def test_float32_io_decides_like_fp64(name, oracle_lib):
    import torch
    L = E.lanes(name)
    g = engine_step(name, L, auto_reset=True)
    h = engine_step(name, L, io_dtype=torch.float32, auto_reset=True)
    for k in ("flag", "done", "time", "episode", "state"):
        bad = g[k] != h[k]
        bad = bad.any(axis=1) if bad.ndim == 2 else bad
        assert not bad.any(), (name, k, int(bad.sum()), _where(L, bad))
    for k in ("obs", "next_obs", "reset_obs", "reward"):
        assert np.array_equal(h["raw_" + k], g["raw_" + k].astype(np.float32)), (name, k)


@pytest.mark.parametrize("name", E.NAMES)
def test_fp32_parked_and_time_lanes_follow_the_float32_rule(name, oracle_lib):
    """fp32 state compared with thresholds rounded to float32, time in float64: the flag of every parked, priority and
    time lane equals the float32 restatement on the engine's own post-step state, the post-step time equals the fp64
    oracle's bit for bit, and parked states keep their float32 bits."""
    import torch
    L = E.lanes(name, np.float32)
    p = E.host(name)._params
    g = engine_step(name, L, dtype=torch.float32)
    o = E.oracle_step(name, L.state, L.time, L.action)
    assert np.array_equal(g["time"], o["time"]), name
    want = E.rule_flag(name, p, L.state, g["state"], g["time"], np.float32)
    bad = g["flag"] != want
    assert not bad.any(), (name, int(bad.sum()), _where(L, bad))
    assert np.array_equal(g["done"], (g["flag"] != 0).astype(np.uint8))
    moving = name in ("cartpole_angleonly_ppo2", "fas", "fas_ppo2", "fas_discrete")
    parked = np.isin(L.kind, ["parked", "priority"] + ([] if moving else ["time"])) & ~np.isin(L.label, ["phi_hi", "phi_lo"])
    moved = np.any(g["raw_state"][parked] != L.state[parked].astype(np.float32), axis=1)
    assert not moved.any(), (name, _where(_sel(L, parked), moved))


@pytest.mark.parametrize("mode", ["fp64", "io32", "fp32"])
@pytest.mark.parametrize("name", E.NAMES)
def test_rollout_kernel_writes_the_bits_of_single_steps(name, mode):
    """the same edge batch for three steps (auto-reset on, so the terminal lanes restart from Philox draws): through
    three step launches and through one b200env_rollout launch -- every output row, the state, time, episode counter
    and the policy observation have the same bits."""
    import torch
    L = E.lanes(name, np.float32 if mode == "fp32" else np.float64)
    n, T = len(L.time), 3
    dtype = torch.float32 if mode == "fp32" else torch.float64
    io = torch.float32 if mode == "io32" else None
    e1, e2 = _env(name, n, dtype, io, True), _env(name, n, dtype, io, True)
    _inject(e1, L)
    _inject(e2, L)
    iod = e1.io_dtype
    A, S = e1._ad, e1._od
    a = torch.from_numpy(np.ascontiguousarray(np.repeat(L.action.T[None], T, 0))).to("cuda", iod)
    z = lambda *s, dt=iod: torch.zeros(*s, dtype=dt, device="cuda")
    bufs = [dict(obs=z(T, S, n), next_obs=z(T, S, n), reward=z(T, n), done=z(T, n, dt=torch.uint8),
                 flag=z(T, n, dt=torch.int32)) for _ in range(2)]
    for t in range(T):
        e1.step_into(a[t], obs=bufs[0]["obs"][t], next_obs=bufs[0]["next_obs"][t], reward=bufs[0]["reward"][t],
                     done=bufs[0]["done"][t], flag=bufs[0]["flag"][t])
    e2.rollout_into(T, a, **bufs[1])
    torch.cuda.synchronize()
    for k in bufs[0]:
        assert torch.equal(bufs[0][k], bufs[1][k]), (name, mode, k)
    assert torch.equal(e1._state, e2._state) and torch.equal(e1._time, e2._time), (name, mode)
    assert torch.equal(e1._episode, e2._episode) and torch.equal(e1.policy_state, e2.policy_state), (name, mode)
    assert int(bufs[0]["done"].sum()) > 0
