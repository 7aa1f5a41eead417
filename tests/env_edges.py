"""Edge lanes of the small env families: states placed on, and a few ulps around, every threshold a step decides on.

A decision of an env step (terminal flag, clamp, angle wrap, time-out, sub-step count, reward branch) compares a value
with a threshold, so one ulp at the threshold changes the flag, the reward by up to several hundred, the bootstrap mask of
GAE and whether the instance auto-resets.  Random trajectories reach a threshold only by chance; these lanes sit on it.

Three kinds of lanes, each `Edge` yielding a block of them:
  parked   the step leaves the state bit-unchanged (zero velocities and action), the decisive value is scanned over the
           doubles around its threshold: outputs must equal the C oracle's bit for bit.
  time     the pre-step time is scanned so that the post-step time lands on time_max and its neighbours, or so that the
           `while time < tt` loop of the sub-stepped families flips between 10 and 11 sub-steps.
  cross    live states whose trajectory crosses the edge inside the step: one pre-state coordinate is bisected with the
           oracle down to the adjacent pair of doubles where its decision flips, then scanned +-64 ulps around it.  The
           engine's flag must equal the reference rule (`rule_flag`) applied to the engine's OWN post-step state.
`priority` blocks are parked or time lanes where several conditions fire at once; they pin each family's flag order.
"""
from __future__ import annotations

import functools
from dataclasses import dataclass, field
from fractions import Fraction
from typing import Callable, Optional

import numpy as np

from helpers import env_specs

NAMES = ["cartpole", "cartpole_angleonly_env", "cartpole_angleonly_ppo2", "fas", "fas_ppo2", "fas_discrete", "soi",
         "soi_dppo2", "ballbalancer", "twolink", "ugv_forward", "ugv_bidirectional", "ugvo", "ugvo_dppo2"]
UGV_NAMES = ("ugv_forward", "ugv_bidirectional")
# UGVForwardObstacleAvoidance: variant 0 (the env, dt 0.1) and variant 1 (the PPO2 / DPPO2 demo copy, dt 0.05); flags
# 1 bounds, 2 time-out, 3 success, 4 collision
UGVO_NAMES = ("ugvo", "ugvo_dppo2")
# the reference loops `while time < tt` in sub-steps of dt / 10: 10 or 11 of them, decided by the rounding of time
SUBSTEP_NAMES = {"cartpole", "cartpole_angleonly_env", "fas", "fas_ppo2", "ballbalancer"}
# success tests on a Euclidean norm: CartPole's Python `sqrt(a*a + b*b + ...)`, the others np.linalg.norm
NORM_EDGES = [("cartpole", "success"), ("cartpole_angleonly_ppo2", "success"), ("soi", "success"), ("twolink", "success"),
              ("ugv_forward", "success"), ("ugv_bidirectional", "success"), ("ugvo", "success"), ("ugvo_dppo2", "success")]
TIME = -1          # Edge.coord of the pre-step time
SEED = 20261021    # Philox seed of the auto-resets (both sides)


# ------------------------------------------------------------------------------------------------------ float bits
def _ord(x, dt=np.float64):
    """doubles (floats) -> integers in the same order, adjacent values one apart (-0.0 and +0.0 both map to 0)."""
    it, mag = (np.int64, 0x7FFFFFFFFFFFFFFF) if dt == np.float64 else (np.int32, 0x7FFFFFFF)
    i = np.asarray(x, dt).view(it)
    return np.where(i < 0, -(i & it(mag)), i).astype(np.int64)


def _unord(o, dt=np.float64):
    it, sign = (np.int64, np.int64(-0x8000000000000000)) if dt == np.float64 else (np.int32, np.int32(-0x80000000))
    o = np.asarray(o, np.int64).astype(it)
    return np.where(o < 0, (-o) | sign, o).astype(it).view(dt)


def ulps(x, k, dt=np.float64):
    return _unord(_ord(x, dt) + k, dt)


# ------------------------------------------------------------------------------------------------------ exact fma
def _round_to(fr: Fraction, dt):
    """correctly rounded (to nearest, ties to even) conversion of an exact rational to float64 / float32."""
    if dt == np.float64:
        return float(fr)  # int / int true division is correctly rounded
    c = np.float32(float(fr))
    best = None
    for v in (np.nextafter(c, np.float32(-np.inf)), c, np.nextafter(c, np.float32(np.inf))):
        d = abs(Fraction(float(v)) - fr)
        key = (d, int(np.asarray(v).view(np.int32)) & 1)
        if best is None or key < best[0]:
            best = (key, v)
    return best[1]


def fma_exact(a, b, c, dt=np.float64):
    """fl(a * b + c) with one rounding, elementwise (Python 3.12 has no math.fma)."""
    a, b, c = (np.asarray(v, dt).ravel() for v in (a, b, c))
    out = np.empty(a.shape, dt)
    for i in range(a.size):
        if not (np.isfinite(a[i]) and np.isfinite(b[i]) and np.isfinite(c[i])):
            out[i] = a[i] * b[i] + c[i]
        else:
            out[i] = _round_to(Fraction(float(a[i])) * Fraction(float(b[i])) + Fraction(float(c[i])), dt)
    return out


def np_norm2(a, b, dt=np.float64):
    """np.linalg.norm((a, b)) as numpy computes it (FMA-accumulated ddot): sqrt(fma(b, b, a * a))."""
    a, b = np.asarray(a, dt), np.asarray(b, dt)
    return np.sqrt(fma_exact(b, b, a * a, dt)).reshape(a.shape)


# ------------------------------------------------------------------------------------------------------ reference rules
def rule_flag(name, p, pre, post, time, dt=np.float64):
    """terminal flag of the reference's is_Terminal() on a post-step state ([lanes, fields]), evaluated in `dt` with the
    thresholds rounded to `dt` like the kernels' `(T)p.x`, every product and sum rounded on its own in the oracle's
    order (numpy does not contract), np.linalg.norm in its FMA form.  `pre` is only read by BallBalancer1D, whose
    is_success() sees the previous step's error."""
    T = lambda v: dt(v)
    s = np.asarray(post, dt)
    time = np.asarray(time, np.float64)
    tout = time > p.time_max
    flag = np.zeros(len(s), np.int32)
    if name.startswith("cartpole"):
        th, dth, x, dx = s[:, 0], s[:, 1], s[:, 2], s[:, 3]
        angle = (th > T(p.theta_term_hi)) | (th < T(p.theta_term_lo))
        eth, ex = T(0) - th, T(0) - x
        if p.variant == 0:  # every test runs, the last true one wins
            flag[angle] = 1
            flag[(x > T(p.x_max)) | (x < -T(p.x_max))] = 2
            flag[tout] = 3
            flag[np.sqrt(ex * ex + dx * dx + eth * eth + dth * dth) < T(1e-2)] = 4
        elif p.variant == 1:  # the first true test returns
            flag[:] = np.where(angle, 1, np.where(tout, 3, 0))
        else:
            flag[angle] = 1
            flag[tout] = 3
            flag[np.sqrt(eth * eth + dth * dth) < T(1e-2)] = 4
    elif name.startswith("fas_discrete"):
        th = s[:, 0]
        flag[:] = np.where((th > T(p.theta_out)) | (th < -T(p.theta_out)), 1, np.where(tout, 2, 0))
    elif name.startswith("fas"):
        th = s[:, 0]
        flag[th > T(p.theta_term_hi)] = 1
        flag[th < T(p.theta_term_lo)] = 2
        flag[tout] = 3
    elif name.startswith("soi"):
        x, y, vx, vy = s[:, 0], s[:, 1], s[:, 2], s[:, 3]
        adm = T(p.admissible_error)
        out = (x > T(p.map_x) + adm) | (x < T(0) - adm) | (y > T(p.map_y) + adm) | (y < T(0) - adm)
        flag[out] = 1
        flag[tout] = 2
        if p.success_terminal:
            e_pos = np_norm2(T(p.target_x) - x, T(p.target_y) - y, dt)
            flag[(e_pos <= T(0.05)) & (np_norm2(vx, vy, dt) < T(0.05))] = 3
    elif name == "ballbalancer":
        pos, vel, th = s[:, 0], s[:, 1], s[:, 2]
        err = np.asarray(pre, dt)[:, 3]
        succ = (np.abs(err) <= T(0.001)) & (np.abs(vel) <= T(0.005)) & (np.abs(th) <= T(p.deg1))
        flag[:] = np.where((pos < -T(p.L)) | (pos > T(p.L)), 1, np.where(tout, 2, np.where(succ, 3, 0)))
    elif name == "twolink":
        en, wn = np_norm2(s[:, 4], s[:, 5], dt), np_norm2(s[:, 2], s[:, 3], dt)
        flag[:] = np.where(tout, 2, np.where((en <= T(p.miss)) & (wn <= T(p.omega_ok)), 3, 0))
    elif name in UGVO_NAMES:  # is_Terminal: every test runs, the last true one wins
        x, y = s[:, 0], s[:, 1]
        flag[(x > T(p.map_x)) | (x < T(0)) | (y > T(p.map_y)) | (y < T(0))] = 1
        flag[tout] = 2
        flag[_ugvo_success(p, s, dt)] = 3
        flag[_ugvo_collided(p, s, dt)] = 4
    elif name in UGV_NAMES:
        x, y, vel = s[:, 0], s[:, 1], s[:, 2]
        flag[(x > T(p.map_x)) | (x < T(0)) | (y > T(p.map_y)) | (y < T(0))] = 1
        flag[tout] = 2
        dx, dy = T(p.target_x) - x, T(p.target_y) - y
        e = np_norm2(dx, dy, dt)
        if p.bidirectional:  # e = sign(d) * |e|: a target abeam (d == 0) counts as reached, 0.3 m away or not
            phi = s[:, 3]
            e = np.where(np.cos(phi) * dx + np.sin(phi) * dy == 0, T(0), e)
        flag[(np.abs(e) <= T(0.05)) & (np.abs(vel) < T(0.01))] = 3
    else:
        raise KeyError(name)
    return flag


def _ugvo_success(p, s, dt=np.float64, norm=None):
    """is_success :423-429 (variant 0) / demo copy :421-427 (variant 1, no omega test) on states [lanes, 56] in `dt`."""
    T = dt
    s = np.asarray(s, dt)
    norm = norm or (lambda a, b: np_norm2(a, b, dt))
    ok = (norm(s[:, 5] - s[:, 0], s[:, 6] - s[:, 1]) <= T(0.05)) & (np.abs(s[:, 2]) < T(0.01))
    return ok & (np.abs(s[:, 4]) < T(0.01)) if p.variant == 0 else ok


def _ugvo_collided(p, s, dt=np.float64):
    """collision_check :261-272: some circle k < n_obs with |pos - centre| <= r_k + r_vehicle."""
    s = np.asarray(s, dt)
    hit = np.zeros(len(s), bool)
    for k in range(16):
        cx, cy, r = s[:, 8 + 3 * k], s[:, 9 + 3 * k], s[:, 10 + 3 * k]
        hit |= (k < s[:, 7]) & (np_norm2(s[:, 0] - cx, s[:, 1] - cy, dt) <= r + dt(p.r_vehicle))
    return hit


def contracted_success(name, p, post):
    """The success test of `name` evaluated the other way round -- CartPole's sum of squares contracted into FMAs the way
    nvcc does it (mul, then fma per further term), the np.linalg.norm envs with plain a*a + b*b -- to show that the
    crossing lanes tell the two evaluations apart."""
    s = np.asarray(post, np.float64)
    sq = lambda a, b: b * b + a * a
    if name == "cartpole":
        ex, eth = 0.0 - s[:, 2], 0.0 - s[:, 0]
        acc = ex * ex
        for v in (s[:, 3], eth, s[:, 1]):
            acc = fma_exact(v, v, acc)
        return np.sqrt(acc) < 1e-2
    if name == "cartpole_angleonly_ppo2":
        eth = 0.0 - s[:, 0]
        return np.sqrt(fma_exact(s[:, 1], s[:, 1], eth * eth)) < 1e-2
    if name == "soi":
        return (np.sqrt(sq(p.target_x - s[:, 0], p.target_y - s[:, 1])) <= 0.05) & (np.sqrt(sq(s[:, 2], s[:, 3])) < 0.05)
    if name == "twolink":
        return (np.sqrt(sq(s[:, 4], s[:, 5])) <= p.miss) & (np.sqrt(sq(s[:, 2], s[:, 3])) <= p.omega_ok)
    if name in UGVO_NAMES:
        return _ugvo_success(p, s, norm=lambda a, b: np.sqrt(sq(a, b)))
    if name in UGV_NAMES:
        return (np.sqrt(sq(p.target_x - s[:, 0], p.target_y - s[:, 1])) <= 0.05) & (np.abs(s[:, 2]) < 0.01)
    raise KeyError(name)


def reference_success(name, p, post):
    """the success test of `name` in the reference's evaluation order (the flag-4 / flag-3 condition alone)."""
    s = np.asarray(post, np.float64)
    if name == "cartpole":
        ex, eth = 0.0 - s[:, 2], 0.0 - s[:, 0]
        return np.sqrt(ex * ex + s[:, 3] * s[:, 3] + eth * eth + s[:, 1] * s[:, 1]) < 1e-2
    if name == "cartpole_angleonly_ppo2":
        eth = 0.0 - s[:, 0]
        return np.sqrt(eth * eth + s[:, 1] * s[:, 1]) < 1e-2
    if name == "soi":
        return (np_norm2(p.target_x - s[:, 0], p.target_y - s[:, 1]) <= 0.05) & (np_norm2(s[:, 2], s[:, 3]) < 0.05)
    if name == "twolink":
        return (np_norm2(s[:, 4], s[:, 5]) <= p.miss) & (np_norm2(s[:, 2], s[:, 3]) <= p.omega_ok)
    if name in UGVO_NAMES:
        return _ugvo_success(p, s)
    if name in UGV_NAMES:
        return (np_norm2(p.target_x - s[:, 0], p.target_y - s[:, 1]) <= 0.05) & (np.abs(s[:, 2]) < 0.01)
    raise KeyError(name)


def _angleonly_reward(p, cur0, nxt0, flag):
    """CartPoleAngleOnly.py:188-208: every branch constant, so the reward is exact given the observations."""
    deg = lambda o: np.abs(o / p.static_gain * p.theta_max * 180. / np.pi)
    ce, ne = deg(np.asarray(cur0, np.float64)), deg(np.asarray(nxt0, np.float64))
    r = np.where(ne > ce, -2.0, np.where(ne == ce, 0.0, 2.0))
    r = r + np.where((ce <= 0.5) & (ne <= 0.5), 5.0, 0.0)
    return r + np.where(flag == 1, -100.0, np.where(flag == 3, 500.0, 0.0))


def _ugv_reward(p, post, flag):
    """UGVForward.py / UGVBidirectional.py get_reward on a post-step state, heading error from numpy's atan2; also returns
    the lanes where that reward is well defined against the kernel's (no ulp-level choice of atan2 or of sign(d) in it)."""
    s = np.asarray(post, np.float64)
    x, y, vel, phi, om = s.T
    dx, dy = p.target_x - x, p.target_y - y
    e = np_norm2(dx, dy)
    c, sn = np.cos(phi), np.sin(phi)
    guard = (np_norm2(dx, dy) < 1e-4) | (np_norm2(c, sn) < 1e-4)
    ephi = np.where(guard, 0.0, np.arctan2(c * dy - sn * dx, c * dx + sn * dy))
    ok = np.abs(np.abs(ephi) - np.pi / 2) > 1e-9
    if p.bidirectional:
        d = c * dx + sn * dy
        ok &= np.abs(d) > 1e-9
        e = np.sign(d) * e
        ephi = np.where(ephi >= np.pi / 2, ephi - np.pi, ephi)
        ephi = np.where(ephi <= -np.pi / 2, ephi + np.pi, ephi)
    u = -np.abs(e) * p.Q_pos + -np.abs(vel) * p.Q_vel
    u_phi = np.where(e > 0.1, -np.abs(ephi) * p.Q_phi, 0.0)
    tot = u + u_phi + -np.abs(om) * p.Q_omega
    return tot, ok


def _ugvo_reward(p, out):
    """get_reward :451-467 (variant 0) / demo copy :449-473 (variant 1) from a lane's own outputs (fp64).  Variant 0: the
    heading term from numpy's atan2 and `ok` = lanes where that is well defined against the kernel's; variant 1 has no
    transcendental: r2 / r3 compare the pre- and post-step observations, r4 reads the success rule and the flag.
    Returns (reward, ok, branch code)."""
    s = np.asarray(out["state"], np.float64)
    x, y, vel, phi, om = s[:, :5].T
    dx, dy = s[:, 5] - x, s[:, 6] - y
    err = np_norm2(dx, dy)
    if p.variant == 0:
        c, sn = np.cos(phi), np.sin(phi)
        guard = (err < 1e-4) | (np_norm2(c, sn) < 1e-4)
        ephi = np.where(guard, 0.0, np.arctan2(c * dy - sn * dx, c * dx + sn * dy))
        u_pos, u_vel, u_om = -np.abs(err) * p.Q_pos, -np.abs(vel) * p.Q_vel, -np.abs(om) * p.Q_omega
        u_phi = np.where(err > 0.1, -np.abs(ephi) * p.Q_phi, 0.0)
        u_psi = np.where(out["flag"] == 1, (p.time_max - np.asarray(out["time"], np.float64)) / p.dt * (u_pos + u_vel + u_phi + u_om), 0.0)
        return u_pos + u_vel + u_phi + u_om + u_psi, np.ones(len(s), bool), (err > 0.1).astype(np.int32)
    cur, nxt = np.asarray(out["obs"], np.float64), np.asarray(out["next_obs"], np.float64)
    r1 = -1 - np.abs(om) * 0.1
    r2 = np.where(cur[:, 0] > nxt[:, 0] + 1e-3, 5.0, np.where(1e-3 + cur[:, 0] < nxt[:, 0], -5.0, 0.0))
    a, b = np.abs(cur[:, 1]), np.abs(nxt[:, 1])
    r3 = np.where(a > b + 1e-2, 2.0, np.where(1e-2 + a < b, -2.0, 0.0))
    r4 = np.where(_ugvo_success(p, s), 500.0, np.where(out["flag"] == 4, -300.0, 0.0))
    code = (3 * (np.sign(r2) + 1) + np.sign(r3) + 1).astype(np.int32) + 9 * np.sign(r4).astype(np.int32)
    return r1 + r2 + r3 + r4, np.ones(len(s), bool), code


def reward_branch(name, p, out):
    """the reward branch a lane took, from its own outputs (None: the reward has no branch besides the flag's)."""
    s = np.asarray(out["state"], np.float64)
    if name == "cartpole_angleonly_env":
        return _angleonly_reward(p, out["obs"][:, 0], out["next_obs"][:, 0], out["flag"])
    if name == "ballbalancer":
        return (np.abs(s[:, 3]) <= 0.001) & (np.abs(s[:, 1]) <= 0.005) & (np.abs(s[:, 2]) <= p.deg1)
    if name in UGVO_NAMES:
        return _ugvo_reward(p, out)[2]
    if name in UGV_NAMES:
        return np_norm2(p.target_x - s[:, 0], p.target_y - s[:, 1]) > 0.1
    return None


def rule_extras(name, p, out):
    """Decisions besides the flag, checked on the engine's own outputs (fp64): returns {check: failing-lane mask}."""
    s = np.asarray(out["state"], np.float64)
    bad = {}
    if name == "cartpole_angleonly_env":
        want = _angleonly_reward(p, out["obs"][:, 0], out["next_obs"][:, 0], out["flag"])
        bad["reward branch (ne > ce, ne == ce, ce/ne <= 0.5 deg)"] = out["reward"] != want
    elif name == "fas_discrete":
        bad["|theta| <= theta_max after the clamp"] = np.abs(s[:, 0]) > p.theta_max
        bad["theta_out unreachable after the clamp"] = out["flag"] == 1
    elif name == "ballbalancer":
        succ = (np.abs(s[:, 3]) <= 0.001) & (np.abs(s[:, 1]) <= 0.005) & (np.abs(s[:, 2]) <= p.deg1)
        bad["reward +1000 branch on the new error"] = (out["reward"] > 500) != succ
        bad["vel clamp"] = (s[:, 1] < p.v_min) | (s[:, 1] > p.v_max)
        bad["theta clamp"] = (s[:, 2] < p.theta_min) | (s[:, 2] > p.theta_max)
    elif name == "twolink":
        bad["wrap into [-theta_max, theta_max]"] = (np.abs(s[:, 0]) > p.theta_max) | (np.abs(s[:, 1]) > p.theta_max)
    elif name in UGVO_NAMES:
        bad["phi wrap into [-pi, pi]"] = np.abs(s[:, 3]) > np.pi
        if p.variant == 0:
            bad["vel >= 0 clamp"] = s[:, 2] < 0
        want, ok, _ = _ugvo_reward(p, out)
        if p.variant == 0:   # atan2 in the heading term: within 1e-9 relative
            bad["reward (u_phi above err 0.1, u_psi on flag 1)"] = ok & (np.abs(out["reward"] - want) > 1e-9 * np.maximum(1.0, np.abs(want)))
        else:                # every term a branch constant: bit for bit
            bad["reward r1 + r2 + r3 + r4"] = out["reward"] != want
    elif name in UGV_NAMES:
        bad["phi wrap into [-pi, pi]"] = np.abs(s[:, 3]) > np.pi
        if not p.bidirectional:
            bad["vel >= 0 clamp"] = s[:, 2] < 0
        want, ok = _ugv_reward(p, s, out["flag"])
        nf = out["flag"] != 1
        bad["reward branch e > 0.1"] = ok & nf & (np.abs(out["reward"] - want) > 1e-9 * np.maximum(1.0, np.abs(want)))
    return bad


# ------------------------------------------------------------------------------------------------------ env plumbing
def host(name):
    cls, kw = env_specs()[name]
    return cls(n_envs=1, host_only=True, **kw)


def oracle_step(name, st, tm, act, auto_reset=False, seed=SEED):
    """one step of the C oracle on lanes-first arrays -> dict of lanes-first outputs (state / time after the step)."""
    from oracle import oracle
    from reinforcementlearningplatform_b200 import _lib
    cls, kw = env_specs()[name]
    h = cls(n_envs=1, host_only=True, **kw)
    L = len(tm)
    sf, od, ad, dd = _lib.dims(cls.ENV_ID, h.VARIANT)
    o = oracle.OracleEnv(cls.ENV_ID, h._params, L, sf, od, ad, dd, seed=seed, auto_reset=auto_reset, nthreads=4)
    o.state[:] = np.asarray(st, np.float64).T
    o.time[:] = tm
    o.step(np.ascontiguousarray(np.asarray(act, np.float64).T))
    return dict(obs=o.obs.T.copy(), next_obs=o.next_obs.T.copy(), reset_obs=o.reset_obs.T.copy(), reward=o.reward.copy(),
                done=o.done.copy(), flag=o.flag.copy(), state=o.state.T.copy(), time=o.time.copy(),
                substeps=o.substeps.copy(), episode=o.episode.copy())


# ------------------------------------------------------------------------------------------------------ edges
@dataclass
class Edge:
    label: str
    kind: str                       # parked | time | cross | priority
    coord: int                      # state field scanned / bisected, or TIME
    state: np.ndarray               # [B, F] base pre-states
    time: np.ndarray                # [B]
    action: np.ndarray              # [B, A] (float32-representable)
    pred: Callable                  # oracle outputs -> bool [lanes]: the decision this edge is about
    lo: Optional[np.ndarray] = None  # bisection bracket of the coordinate (cross / bisected parked edges)
    hi: Optional[np.ndarray] = None
    center: Optional[np.ndarray] = None  # scan centre when there is no bracket
    K: int = 8                      # lanes at -K .. K ulps of the flip / centre
    derive: Optional[Callable] = None  # (state [L, F], dtype) -> None: fields that follow the scanned one
    cover: bool = True              # coverage: both sides of `pred` within 2 ulps of the flip


@dataclass
class Lanes:
    state: np.ndarray
    time: np.ndarray
    action: np.ndarray
    label: np.ndarray
    kind: np.ndarray
    k: np.ndarray                   # ulp offset from the flip (first lane on the far side = 0) or from the centre
    blocks: list = field(default_factory=list)  # (Edge, slice)


def _place(e, vals, reps, dt=np.float64):
    st = np.repeat(e.state, reps, axis=0).astype(np.float64)
    tm = np.repeat(e.time, reps).astype(np.float64)
    if e.coord == TIME:
        tm[:] = vals
    else:
        st[:, e.coord] = vals
    if dt == np.float32:
        st = st.astype(np.float32).astype(np.float64)
    if e.derive is not None:
        e.derive(st, dt)
    return st, tm


def _run_pred(name, e, vals):
    st, tm = _place(e, vals, 1)
    return e.pred(oracle_step(name, st, tm, e.action)), st


def _flip(name, e):
    """vectorised bisection over the doubles: the adjacent pair (lo, hi) where e.pred changes.  Returns the edge restricted
    to the bases whose bracket ends decide differently, ord(hi) and the direction (+-1) from lo to hi in that order."""
    lo, hi = _ord(e.lo), _ord(e.hi)
    plo = _run_pred(name, e, _unord(lo))[0]
    phi = _run_pred(name, e, _unord(hi))[0]
    keep = plo != phi
    lo, hi, plo = lo[keep], hi[keep], plo[keep]
    sub = Edge(**{**e.__dict__, "state": e.state[keep], "time": e.time[keep], "action": e.action[keep]})
    for _ in range(80):
        if not np.any(np.abs(hi - lo) > 1):
            break
        mid = lo + (hi - lo) // 2
        pm = _run_pred(name, sub, _unord(mid))[0]
        lo = np.where(pm == plo, mid, lo)
        hi = np.where(pm == plo, hi, mid)
    assert np.all(np.abs(hi - lo) == 1), (name, e.label)
    return sub, hi, hi - lo


def _expand(name, e, dt=np.float64):
    sd = np.float64 if e.coord == TIME else dt   # the scan's step: time is float64 in every mode
    if e.lo is not None and dt == np.float64:
        e, c, sgn = _flip(name, e)
    else:
        c = _ord(e.center if sd == np.float64 else np.asarray(e.center, np.float64).astype(np.float32), sd)
        sgn = np.ones_like(c)
    ks = np.arange(-e.K, e.K + 1)
    vals = _unord((c[:, None] + sgn[:, None] * ks[None, :]).ravel(), sd).astype(np.float64)
    st, tm = _place(e, vals, len(ks), dt)
    act = np.repeat(e.action, len(ks), axis=0)
    return st, tm, act, np.tile(ks, len(c))


def _mk(B, F, A):
    return np.zeros((B, F)), np.zeros(B), np.zeros((B, A))


def _uniform(rng, lo, hi, B):
    return rng.uniform(lo, hi, B)


def _f32(a):
    return np.asarray(a, np.float64).astype(np.float32).astype(np.float64)


def _time_edges(name, p, st0, act0, loops):
    """time lanes: post-step time on time_max and its neighbours; sub-step count flips (10 | 11) for the looped envs."""
    flagt = {"cartpole": 3, "cartpole_angleonly_env": 3, "cartpole_angleonly_ppo2": 3, "fas": 3, "fas_ppo2": 3}.get(name, 2)
    B = 1
    # bisected: where the sub-step count is 11 the post-step time reaches time_max from time_max - 1.1 dt, not - dt
    edges = [Edge("time_max", "time", TIME, st0[None, :].copy(), np.zeros(B), act0[None, :].copy(),
                  pred=lambda o, f=flagt: o["flag"] == f, lo=np.array([p.time_max - 1.5 * p.dt]),
                  hi=np.array([p.time_max - 0.5 * p.dt]), K=256)]
    if loops:
        # the count is constant over long runs of pre-step times (it changes mostly with the binade of time): brackets
        # around the changes on a fine grid of [0, time_max], bisected to the doubles where it flips
        grid = np.linspace(0.0, p.time_max, 20001)
        n = len(grid)
        sub = oracle_step(name, np.repeat(st0[None, :], n, 0), grid, np.repeat(act0[None, :], n, 0))["substeps"]
        at = np.nonzero(np.diff(sub))[0]
        at = at[np.linspace(0, len(at) - 1, min(24, len(at))).astype(int)]
        B = len(at)
        edges.append(Edge("substeps", "time", TIME, np.repeat(st0[None, :], B, 0), grid[at], np.repeat(act0[None, :], B, 0),
                          pred=lambda o: o["substeps"] == 11, lo=grid[at], hi=grid[at + 1], K=24))
    return edges


UGVO_TARGET = (2.5, 2.5)
# Circles for the pose-level UGV-FOA lanes.  A lane carries those that lie out of laser range of its pose by 0.5 m (more
# than any step moves), so the in-range list is built and comes out empty: the laser only meets walls, whose ranges do
# not jump with an ulp of the slope.  The collision blocks add one circle of their own.
_UGVO_FAR = ((0.4, 0.4, 0.3), (4.6, 0.4, 0.25), (0.4, 4.6, 0.35), (4.6, 4.6, 0.2), (2.5, 0.3, 0.2), (2.5, 4.7, 0.25),
             (0.3, 2.5, 0.2), (4.7, 2.5, 0.3))


def ugvo_row(p, x, y, vel=0.0, phi=0.3, omega=0.0, near=(), target=UGVO_TARGET):
    """one UGV-FOA state [56]: pose, target, the circles `near` first, then the far ones (headings near 0.3 keep every
    ray at least 2 degrees off the vertical)."""
    s = np.zeros(56)
    s[:7] = x, y, vel, phi, omega, target[0], target[1]
    circ = list(near) + [c for c in _UGVO_FAR if np.hypot(c[0] - x, c[1] - y) > p.laser_dis + c[2] + 0.5]
    assert len(circ) >= 1
    s[7] = len(circ)
    for k, c in enumerate(circ):
        s[8 + 3 * k:11 + 3 * k] = c
    return s


def _ugvo_rows(p, x, y, vel, phi, omega, target=UGVO_TARGET):
    return np.stack([ugvo_row(p, *v, target=target) for v in zip(*np.broadcast_arrays(x, y, vel, phi, omega))])


def _ugvo_edges(name, p, rng):
    """the pose-level edges of UGVForwardObstacleAvoidance (variant 0 and the demo copy, variant 1)."""
    E = []
    flag_is = lambda f: (lambda o: o["flag"] == f)
    tx, ty = UGVO_TARGET
    v = p.variant
    B, A = 32, 2
    z1, a0 = np.zeros(1), np.zeros((1, A))
    late = np.array([p.time_max - p.dt / 2])   # the post-step time is past time_max
    box = [("x_hi", 0, p.map_x), ("x_lo", 0, 0.0), ("y_hi", 1, p.map_y), ("y_lo", 1, 0.0)]
    for lab, c, thr in box:
        xy = [tx, ty]
        xy[c] = thr
        s = ugvo_row(p, *xy)
        E.append(Edge(lab, "parked", c, s[None], z1, a0, flag_is(1), center=np.array([thr])))
        E.append(Edge(lab + "+time", "priority", c, s[None], late, a0, flag_is(2), center=np.array([thr]), cover=False))
    for lab, thr in (("phi_hi", np.pi), ("phi_lo", -np.pi)):
        s = ugvo_row(p, 1.0, 1.0, phi=thr)
        E.append(Edge(lab, "parked", 3, s[None], z1, a0, lambda o, t=thr: o["state"][:, 3] * t < 0, center=np.array([thr])))
    s = ugvo_row(p, tx - 0.05, ty)
    E.append(Edge("success_parked", "parked", 0, s[None], z1, a0, flag_is(3), center=np.array([tx - 0.05])))
    sd = np.stack([ugvo_row(p, tx - 0.03, ty - 0.04, phi=1.0), ugvo_row(p, tx + 0.04, ty + 0.03, phi=-2.0)])
    E.append(Edge("success_parked_diag", "parked", 1, sd, np.zeros(2), np.zeros((2, A)), flag_is(3),
                  lo=sd[:, 1] - np.sign(sd[:, 1] - ty) * 0.005, hi=sd[:, 1] + np.sign(sd[:, 1] - ty) * 0.005))
    E.append(Edge("success+time", "priority", 0, s[None], late, a0, flag_is(3), center=np.array([tx - 0.05])))
    # err exactly fl(0.05): x = 2^-10 and target x = 2^-10 + fl(0.05) (the sum and the difference are exact; the target's
    # ulps are err's, so the scan of the target moves err one ulp at a time)
    g = 2.0 ** -10
    s = ugvo_row(p, g, ty, target=(g + 0.05, ty))
    E.append(Edge("success_parked_exact", "parked", 5, s[None], z1, a0, flag_is(3), center=np.array([g + 0.05])))
    s = ugvo_row(p, tx - 1e-4, ty)   # vector_rad_oriented's `norm < 1e-4` guard: ephi (obs 2) == 0
    E.append(Edge("ephi_guard", "parked", 0, s[None], z1, a0, lambda o: o["next_obs"][:, 2] != 0,
                  lo=np.array([tx - 2e-4]), hi=np.array([tx])))
    if v == 0:   # reward branch err > 0.1 (heading error 0.5 rad: u_phi = -1)
        s = ugvo_row(p, tx - 0.1, ty, phi=0.5)
        E.append(Edge("reward_e_0.1", "parked", 0, s[None], z1, a0, lambda o: o["reward"] < -0.5, center=np.array([tx - 0.1])))
    # collision at |pos - centre| == r + r_vehicle: the centre's x bisected to the flip; with several flags at once the
    # collision must win over success + time-out and over bounds
    R = 0.3 + p.r_vehicle
    for lab, kind, (x, y), ang, tm, cov in (("collision", "parked", (1.5, 2.5), 0.0, 0.0, True),
                                            ("collision_diag", "parked", (1.5, 2.5), 0.7, 0.0, True),
                                            ("collision+success+time", "priority", (tx - 0.03, ty), 0.0, late[0], True),
                                            ("collision+x_hi", "priority", (p.map_x, ty), np.pi, 0.0, False)):
        cx, cy = x + R * np.cos(ang), y + R * np.sin(ang)
        s = ugvo_row(p, x, y, near=[(cx, cy, 0.3)])
        sg = 1.0 if np.cos(ang) >= 0 else -1.0
        E.append(Edge(lab, kind, 8, s[None], np.array([tm]), a0, flag_is(4), lo=np.array([cx + sg * 0.01]),
                      hi=np.array([cx - sg * 0.01]), cover=cov))
    if v == 1:   # the pose frozen on the PRE-update velocity (vel < 0): -0.0 and +0.0 move, -5e-324 freezes
        frozen = lambda o: o["state"][:, 0] == 2.0
        s, act = ugvo_row(p, 2.0, 2.0, phi=0.3, omega=0.2), np.array([[2.0, 0.5]])

        def neg0(st, dt):
            st[:, 2] = -0.0
        E.append(Edge("frozen_vel", "cross", 2, s[None], z1, act, frozen, center=np.array([0.0]), K=3))
        E.append(Edge("frozen_vel_neg0", "cross", 2, s[None], z1, act, frozen, center=np.array([0.0]), K=0, derive=neg0, cover=False))
        E.append(Edge("frozen_vel_neg", "cross", 2, s[None], z1, act, frozen, center=np.array([-1e-3]), K=2, cover=False))
        s = ugvo_row(p, p.map_x, ty, vel=-0.5, phi=0.3)   # frozen on the border: the flag from the unmoved x
        E.append(Edge("x_hi_frozen", "cross", 0, s[None], z1, np.array([[1.0, 0.5]]), flag_is(1), center=np.array([p.map_x])))
    E += _time_edges(name, p, ugvo_row(p, 1.5, 1.5), np.zeros(A), False)
    # ---- crossing lanes
    for lab, c, thr in box:
        sgn = 1 if lab.endswith("hi") else -1
        head = (0.0 if sgn > 0 else np.pi) if c == 0 else sgn * np.pi / 2
        xy = [np.full(B, tx), np.full(B, ty)]
        xy[c][:] = thr
        st = _ugvo_rows(p, xy[0], xy[1], rng.uniform(0.5, 2.5, B), head + rng.uniform(-0.4, 0.4, B), rng.uniform(-1, 1, B))
        act = _f32(rng.uniform(-3, 3, (B, A)))
        E.append(Edge(lab + "_cross", "cross", c, st, np.zeros(B), act, flag_is(1), lo=np.full(B, thr - sgn * 0.2),
                      hi=np.full(B, thr + sgn * 0.01), K=64))
    for lab, sgn in (("phi_hi", 1), ("phi_lo", -1)):   # heading wrap at +-pi after RK4
        st = _ugvo_rows(p, rng.uniform(1.5, 3.5, B), rng.uniform(1.5, 3.5, B), rng.uniform(0, 1, B), 0.0,
                        sgn * rng.uniform(0.5, 3, B))
        act = _f32(rng.uniform(-3, 3, (B, A)))
        E.append(Edge(lab + "_cross", "cross", 3, st, np.zeros(B), act, lambda o, s=sgn: s * o["state"][:, 3] < 0,
                      lo=np.full(B, sgn * (np.pi - 0.2)), hi=np.full(B, sgn * np.pi), K=64))
    # success on err <= 0.05 (np.linalg.norm's FMA form), crossed by x; small velocity and rate.  A target near the
    # corner (0, 0): an ulp of x there moves err by a few of its own ulps, so scans land on the threshold
    BS, g = 256, 0.25
    ang = rng.uniform(0, 2 * np.pi, BS)
    om = rng.uniform(-0.005, 0.005, BS) if v == 0 else rng.uniform(-0.5, 0.5, BS)
    st = _ugvo_rows(p, g, g + 0.04 * np.sin(ang), rng.uniform(0, 0.005, BS), rng.uniform(-np.pi, np.pi, BS), om, (g, g))
    act = _f32(np.stack([rng.uniform(-0.03, 0.03, BS), rng.uniform(-0.02, 0.02, BS)], 1))
    E.append(Edge("success", "cross", 0, st, np.zeros(BS), act, flag_is(3), lo=np.full(BS, g), hi=np.full(BS, g + 0.1), K=16))
    # success on |vel| < 0.01, crossed by the pre-step velocity (at the target: err stays ~vel dt)
    st = _ugvo_rows(p, tx, ty, 0.0, rng.uniform(-np.pi, np.pi, B), 0.0)
    act = _f32(np.stack([rng.uniform(-0.05, 0.05, B), np.zeros(B)], 1))
    E.append(Edge("success_vel", "cross", 2, st, np.zeros(B), act, flag_is(3), lo=np.zeros(B), hi=np.full(B, 0.03), K=64))
    if v == 0:   # success on |omega| < 0.01 (variant 0 only), crossed by the pre-step rate, both signs
        for lab, sgn in (("success_omega_pos", 1), ("success_omega_neg", -1)):
            st = _ugvo_rows(p, tx - 0.02, ty, 0.0, rng.uniform(-np.pi, np.pi, B), 0.0)
            act = _f32(np.stack([np.zeros(B), rng.uniform(-0.05, 0.05, B)], 1))
            E.append(Edge(lab, "cross", 4, st, np.zeros(B), act, flag_is(3), lo=np.zeros(B), hi=np.full(B, sgn * 0.03), K=64))
        st = _ugvo_rows(p, tx - 0.1, ty, rng.uniform(0.05, 0.3, B), rng.uniform(0.4, 0.8, B), 0.0)
        act = _f32(rng.uniform(-0.5, 0.5, (B, A)))
        E.append(Edge("reward_e_0.1_cross", "cross", 0, st, np.zeros(B), act, lambda o: o["reward"] < -0.5,
                      lo=np.full(B, tx - 0.2), hi=np.full(B, tx - 0.02), K=64))
        st = _ugvo_rows(p, rng.uniform(1.5, 3.5, B), rng.uniform(1.5, 3.5, B), 0.0, rng.uniform(-3, 3, B), 0.0)
        act = _f32(np.stack([rng.uniform(-3, -0.5, B), rng.uniform(-3, 3, B)], 1))
        E.append(Edge("vel_clamp", "cross", 2, st, np.zeros(B), act, lambda o: o["state"][:, 2] == 0,
                      lo=np.full(B, 0.1), hi=np.zeros(B), K=64))
    else:
        # r2 = +-5 where cur_e - nk0 crosses +-1e-3: heading to / away from the target, crossed by the velocity
        for lab, head, pred in (("reward_r2_pos", 0.0, lambda o: o["reward"] > 0), ("reward_r2_neg", np.pi, lambda o: o["reward"] < -3)):
            st = _ugvo_rows(p, tx - 1.0, ty, 0.0, head + rng.uniform(-0.2, 0.2, B), 0.0)
            E.append(Edge(lab, "cross", 2, st, np.zeros(B), np.zeros((B, A)), pred, lo=np.full(B, 0.01), hi=np.full(B, 0.08), K=64))
        # r3 = +-2 where |cur1| - |nk1| crosses +-1e-2: moving across the target's bearing, the step's velocity change
        # 0.05 (a - 0.1 vel) crossing 0.015 at vel = 0.1
        for lab, a, lo, hi, pred in (("reward_r3_pos", 0.31, 0.0, 0.2, lambda o: o["reward"] > 0.5),
                                     ("reward_r3_neg", -0.29, 0.0, 0.2, lambda o: o["reward"] < -2)):
            st = _ugvo_rows(p, tx - 1.0, ty, 0.0, np.pi / 2 + rng.uniform(-0.05, 0.05, B), 0.0)
            act = _f32(np.stack([np.full(B, a), np.zeros(B)], 1))
            E.append(Edge(lab, "cross", 2, st, np.zeros(B), act, pred, lo=np.full(B, lo), hi=np.full(B, hi), K=64))
    return E


def _family_edges(name, p, rng):
    """the edge inventory of one family (see the module docstring)."""
    E = []
    flag_is = lambda f: (lambda o: o["flag"] == f)
    B = 32
    # norm-based success edges: a lane lands within an ulp of the threshold only once or twice per base (the sum of
    # squares moves ~2 of its ulps per ulp of CartPole's bisected coordinate, 60 for SOI's position and 300 for the
    # two-link target, whose ulps are those of numbers near 2.5 and 1 while the norm is 0.05 and 0.01): many bases,
    # short scans
    BS = {"soi": 2048, "twolink": 4096}.get(name, 256)
    KS = {"soi": 4, "twolink": 2}.get(name, 16)
    if name.startswith("cartpole"):
        v = p.variant
        F, A = 4, 1
        rest = np.zeros(F)
        if v == 0:
            for lab, sgn in (("x_hi", 1), ("x_lo", -1)):
                s = rest.copy(); s[2] = sgn * p.x_max
                E.append(Edge(lab, "parked", 2, s[None], np.zeros(1), np.zeros((1, A)), flag_is(2), center=np.array([sgn * p.x_max])))
            for lab, sgn in (("success_parked", 1), ("success_parked_neg", -1)):
                s = rest.copy(); s[2] = sgn * 1e-2
                E.append(Edge(lab, "parked", 2, s[None], np.zeros(1), np.zeros((1, A)), flag_is(4), center=np.array([sgn * 1e-2])))
            late = np.array([p.time_max - p.dt / 2])
            s = rest.copy(); s[2] = p.x_max
            E.append(Edge("x_hi+time", "priority", 2, s[None], late, np.zeros((1, A)), flag_is(3), center=np.array([p.x_max]), cover=False))
            s = rest.copy(); s[2] = 1e-2
            E.append(Edge("success+time", "priority", 2, s[None], late, np.zeros((1, A)), flag_is(4), center=np.array([1e-2])))
            E += _time_edges(name, p, np.array([0.0, 0.0, 0.5, 0.0]), np.zeros(A), True)
        elif v == 1:
            E += _time_edges(name, p, np.array([0.0, 0.0, 0.3, 0.0]), np.zeros(A), True)  # parked: ne == ce == 0
        else:
            s = rest.copy()
            E.append(Edge("success+time", "priority", TIME, s[None], np.zeros(1), np.zeros((1, A)), flag_is(4),
                          center=np.array([p.time_max - p.dt]), K=8, cover=False))
            E += _time_edges(name, p, np.array([0.0, 0.5, 0.0, 0.0]), np.zeros(A), False)
        # crossing: angle out through either bound; with a simultaneous time-out the flag order decides (variant 1
        # returns at the angle test, variants 0 and 2 let the time-out win)
        for lab, bound, sgn in (("angle_hi", p.theta_term_hi, 1), ("angle_lo", p.theta_term_lo, -1)):
            for late in (False, True):
                st, tm, act = _mk(B, F, A)
                st[:, 1] = sgn * _uniform(rng, 0.3, 2.0, B)
                st[:, 2] = _uniform(rng, -0.5, 0.5, B) if v == 0 else 0.0
                st[:, 3] = _uniform(rng, -0.5, 0.5, B)
                act[:, 0] = _f32(_uniform(rng, -5, 5, B))
                if late:
                    tm[:] = p.time_max - p.dt / 2
                if late and v != 1:
                    E.append(Edge(lab + "+time", "cross", 0, st, tm, act, flag_is(3), center=np.full(B, bound), K=64, cover=False))
                else:
                    E.append(Edge(lab + ("+time" if late else ""), "cross", 0, st, tm, act, flag_is(1),
                                  lo=bound - sgn * 0.2 * np.ones(B), hi=bound + sgn * 0.01 * np.ones(B), K=64))
        if v == 0:  # angle out while the cart is already beyond x_max: the position test runs later and wins (flag 2)
            for lab, bound, sgn in (("angle_hi+x", p.theta_term_hi, 1), ("angle_lo+x", p.theta_term_lo, -1)):
                st, tm, act = _mk(B, F, A)
                st[:, 1] = sgn * _uniform(rng, 0.3, 2.0, B)
                st[:, 2] = sgn * (p.x_max + _uniform(rng, 0.05, 0.3, B))
                st[:, 3] = sgn * _uniform(rng, 0.0, 0.5, B)
                act[:, 0] = _f32(_uniform(rng, -5, 5, B))
                E.append(Edge(lab, "cross", 0, st, tm, act, flag_is(2), center=np.full(B, bound), K=64, cover=False))
            for lab, sgn in (("x_hi", 1), ("x_lo", -1)):
                st, tm, act = _mk(B, F, A)
                st[:, 0] = _uniform(rng, -0.05, 0.05, B)
                st[:, 3] = sgn * _uniform(rng, 0.5, 2.0, B)
                act[:, 0] = _f32(_uniform(rng, -5, 5, B))
                E.append(Edge(lab + "_cross", "cross", 2, st, tm, act, flag_is(2),
                              lo=sgn * (p.x_max - 0.2) * np.ones(B), hi=sgn * (p.x_max + 0.01) * np.ones(B), K=64))
        if v in (0, 2):
            st, tm, act = _mk(BS, F, A)
            st[:, 0] = _uniform(rng, -3e-3, 3e-3, BS)
            st[:, 1] = _uniform(rng, -3e-3, 3e-3, BS)
            st[:, 3] = _uniform(rng, -3e-3, 3e-3, BS) if v == 0 else 0.0
            act[:, 0] = _f32(_uniform(rng, -0.01, 0.01, BS))
            coord = 2 if v == 0 else 1
            E.append(Edge("success", "cross", coord, st, tm, act, flag_is(4), lo=np.zeros(BS), hi=np.full(BS, 0.05), K=KS))
        if v == 1:  # reward branch `ce <= 0.5 and ne <= 0.5` (degrees), crossed by ne (moving out) and by ce (moving in)
            half = 0.5 * np.pi / 180
            for lab, sgn in (("reward_ne_half_deg", 1), ("reward_ce_half_deg", -1)):
                st, tm, act = _mk(B, F, A)
                st[:, 1] = sgn * _uniform(rng, 0.05, 0.3, B)
                act[:, 0] = _f32(_uniform(rng, -0.5, 0.5, B))
                E.append(Edge(lab, "cross", 0, st, tm, act, lambda o: o["reward"] >= 3,
                              lo=np.full(B, half - 0.01), hi=np.full(B, half + 0.01), K=64))
    elif name.startswith("fas_discrete"):
        F, A = 2, 1
        E += _time_edges(name, p, np.zeros(F), np.zeros(A), False)
        for lab, sgn in (("clamp_hi", 1), ("clamp_lo", -1)):
            st, tm, act = _mk(B, F, A)
            st[:, 1] = sgn * _uniform(rng, 0.2, 2.0, B)
            act[:, 0] = _f32(_uniform(rng, -1.6, 3.0, B))
            clamped = lambda o, s=sgn: o["state"][:, 0] == s * p.theta_max
            E.append(Edge(lab, "cross", 0, st, tm, act, clamped,
                          lo=np.full(B, sgn * (p.theta_max - 0.3)), hi=np.full(B, sgn * p.theta_max), K=64))
    elif name.startswith("fas"):
        F, A = 2, 1
        E += _time_edges(name, p, np.zeros(F), np.zeros(A), True)
        for lab, bound, sgn, f in (("theta_hi", p.theta_term_hi, 1, 1), ("theta_lo", p.theta_term_lo, -1, 2)):
            for late in (False, True):
                st, tm, act = _mk(B, F, A)
                st[:, 1] = sgn * _uniform(rng, 0.3, 2.0, B)
                act[:, 0] = _f32(_uniform(rng, -1.5, 4.0, B))
                if late:
                    tm[:] = p.time_max - p.dt / 2
                if late:  # every test runs, the time-out (last) wins
                    E.append(Edge(lab + "+time", "cross", 0, st, tm, act, flag_is(3), center=np.full(B, bound), K=64, cover=False))
                else:
                    E.append(Edge(lab, "cross", 0, st, tm, act, flag_is(f), lo=np.full(B, bound - sgn * 0.1),
                                  hi=np.full(B, bound + sgn * 0.01), K=64))
    elif name.startswith("soi"):
        F, A = 4, 2
        tx, ty = p.target_x, p.target_y
        box = [("x_hi", 0, p.map_x + p.admissible_error), ("x_lo", 0, 0 - p.admissible_error),
               ("y_hi", 1, p.map_y + p.admissible_error), ("y_lo", 1, 0 - p.admissible_error)]
        for lab, c, thr in box:
            s = np.array([tx, ty, 0.0, 0.0]); s[c] = thr
            E.append(Edge(lab, "parked", c, s[None], np.zeros(1), np.zeros((1, A)), flag_is(1), center=np.array([thr])))
            E.append(Edge(lab + "+time", "priority", c, s[None], np.array([p.time_max - p.dt]), np.zeros((1, A)),
                          flag_is(2), center=np.array([thr]), cover=False))
        succ = flag_is(3)   # dppo2: success is off, the lanes pin that flag 3 never comes
        on = bool(p.success_terminal)
        s = np.array([tx - 0.05, ty, 0.0, 0.0])
        E.append(Edge("success_parked", "parked", 0, s[None], np.zeros(1), np.zeros((1, A)), succ, center=np.array([tx - 0.05]), cover=on))
        sd = np.array([[tx - 0.03, ty - 0.04, 0, 0], [tx + 0.04, ty + 0.03, 0, 0], [tx - 0.01, ty + 0.0499, 0, 0]])
        if on:
            E.append(Edge("success_parked_diag", "parked", 1, sd, np.zeros(3), np.zeros((3, A)), succ,
                          lo=sd[:, 1] - np.sign(sd[:, 1] - ty) * 0.005, hi=sd[:, 1] + np.sign(sd[:, 1] - ty) * 0.005))
        else:
            E.append(Edge("success_parked_diag", "parked", 1, sd, np.zeros(3), np.zeros((3, A)), succ, center=sd[:, 1], cover=False))
        E.append(Edge("success+time", "priority", 0, s[None], np.array([p.time_max - p.dt]), np.zeros((1, A)), succ,
                      center=np.array([tx - 0.05]), cover=on))
        E += _time_edges(name, p, np.array([1.0, 1.0, 0.0, 0.0]), np.zeros(A), False)
        for lab, c, thr in box:
            sgn = 1 if lab.endswith("hi") else -1
            st, tm, act = _mk(B, F, A)
            st[:, 0], st[:, 1] = tx, ty
            st[:, 2 + c] = sgn * _uniform(rng, 0.3, 2.0, B)
            st[:, 3 - c] = _uniform(rng, -1, 1, B)
            act[:] = _f32(rng.uniform(-3, 3, (B, A)))
            E.append(Edge(lab + "_cross", "cross", c, st, tm, act, flag_is(1), lo=np.full(B, thr - sgn * 0.2),
                          hi=np.full(B, thr + sgn * 0.01), K=64))
        if on:
            st, tm, act = _mk(BS, F, A)
            ang = rng.uniform(0, 2 * np.pi, BS)
            st[:, 1] = ty + 0.04 * np.sin(ang)
            st[:, 2] = _uniform(rng, -0.02, 0.02, BS)
            st[:, 3] = _uniform(rng, -0.02, 0.02, BS)
            act[:] = _f32(rng.uniform(-0.3, 0.3, (BS, A)))
            E.append(Edge("success", "cross", 0, st, tm, act, succ, lo=np.full(BS, tx), hi=np.full(BS, tx - 0.1), K=KS))
    elif name == "ballbalancer":
        F, A = 4, 1

        # a parked ball keeps error == target - pos, so that the step rewrites the error with the same bits
        def park_err(st, dt):  # pos from the scanned error
            st[:, 0] = (dt(p.target) - st[:, 3].astype(dt)).astype(np.float64)

        def d(st, dt):  # error from the scanned pos
            st[:, 3] = (dt(p.target) - st[:, 0].astype(dt)).astype(np.float64)
        for lab, sgn in (("pos_hi", 1), ("pos_lo", -1)):
            s = np.array([sgn * p.L, 0, 0, p.target - sgn * p.L])
            E.append(Edge(lab, "parked", 0, s[None], np.zeros(1), np.zeros((1, A)), flag_is(1), center=np.array([sgn * p.L]), derive=d))
            E.append(Edge(lab + "+time", "priority", 0, s[None], np.array([p.time_max - p.dt]), np.zeros((1, A)), flag_is(1),
                          center=np.array([sgn * p.L]), derive=d, cover=False))
        for lab, sgn in (("success_parked", 1), ("success_parked_neg", -1)):
            s = np.array([0, 0, 0, sgn * 0.001])
            E.append(Edge(lab, "parked", 3, s[None], np.zeros(1), np.zeros((1, A)), flag_is(3), center=np.array([sgn * 0.001]),
                          derive=park_err))
        s = np.array([0, 0, 0, 0.0005])
        E.append(Edge("success+time", "priority", TIME, s[None], np.zeros(1), np.zeros((1, A)), flag_is(2),
                      center=np.array([p.time_max - p.dt]), derive=park_err, cover=False))
        E += _time_edges(name, p, np.array([-0.05, 0, 0, p.target + 0.05]), np.zeros(A), True)
        for lab, sgn in (("pos_hi", 1), ("pos_lo", -1)):
            st, tm, act = _mk(B, F, A)
            st[:, 1] = sgn * _uniform(rng, 0.3, 2.0, B)
            st[:, 2] = _uniform(rng, -0.5, 0.5, B)
            act[:, 0] = _f32(_uniform(rng, -3, 3, B))
            E.append(Edge(lab + "_cross", "cross", 0, st, tm, act, flag_is(1), lo=np.full(B, sgn * (p.L - 0.1)),
                          hi=np.full(B, sgn * (p.L + 0.01)), K=64))
        st, tm, act = _mk(BS, F, A)   # success on the previous step's error, crossed by the new velocity
        st[:, 0] = _uniform(rng, -0.02, 0.02, BS)
        st[:, 2] = _uniform(rng, -0.01, 0.01, BS)
        st[:, 3] = _uniform(rng, -0.001, 0.001, BS)
        act[:, 0] = _f32(_uniform(rng, -0.2, 0.2, BS))
        E.append(Edge("success", "cross", 1, st, tm, act, flag_is(3), lo=np.zeros(BS), hi=np.full(BS, 0.01), K=KS))
        for lab, c, thr in (("vel_clamp", 1, p.v_max), ("theta_clamp", 2, p.theta_max)):
            st, tm, act = _mk(B, F, A)
            st[:, 0] = _uniform(rng, -0.05, 0.05, B)
            st[:, 1] = _uniform(rng, 0, 0.5, B)
            st[:, 2] = _uniform(rng, 0.3, 0.7, B)
            act[:, 0] = _f32(_uniform(rng, 0.5, 3.5, B))   # beyond omega_max in some lanes: the action clip
            E.append(Edge(lab, "cross", c, st, tm, act, lambda o, c=c, t=thr: o["state"][:, c] == t,
                          lo=np.full(B, thr - 0.2), hi=np.full(B, thr), K=64))
    elif name == "twolink":
        F, A = 8, 2
        l, bx, by = p.l, p.base_x, p.base_y
        endx = l * np.sin(0.0) + bx + l * np.sin(0.0)
        endy = (-l * np.cos(0.0) + by) + -l * np.cos(0.0)

        def park_err(st, dt):  # arm at rest at theta = 0: the step rewrites err = target - end with the same bits
            T = dt
            ex = T(l) * T(0) + T(bx) + T(l) * T(0)
            ey = (-T(l) * T(1) + T(by)) + -T(l) * T(1)
            st[:, 4] = (st[:, 6].astype(T) - ex).astype(np.float64)
            st[:, 5] = (st[:, 7].astype(T) - ey).astype(np.float64)
        for lab, ang in (("success_parked", 0.0), ("success_parked_diag", 0.9)):
            s = np.zeros(F); s[6], s[7] = endx + p.miss * np.cos(ang), endy + p.miss * np.sin(ang)
            E.append(Edge(lab, "parked", 6, s[None], np.zeros(1), np.zeros((1, A)), flag_is(3),
                          lo=np.array([s[6] + 0.002]), hi=np.array([s[6] - 0.002]), derive=park_err))
        s = np.zeros(F); s[6], s[7] = endx + 0.5 * p.miss, endy
        E.append(Edge("success+time", "priority", TIME, s[None], np.zeros(1), np.zeros((1, A)), flag_is(2),
                      center=np.array([p.time_max - p.dt]), derive=park_err, cover=False))
        s = np.zeros(F); s[6], s[7] = 1.5, 1.5
        E += [Edge("time_max", "time", TIME, s[None], np.zeros(1), np.zeros((1, A)), flag_is(2),
                   lo=np.array([p.time_max - 1.5 * p.dt]), hi=np.array([p.time_max - 0.5 * p.dt]), K=256, derive=park_err)]
        for c in (0, 1):
            for lab, sgn in (("hi", 1), ("lo", -1)):
                st, tm, act = _mk(B, F, A)
                st[:, 1 - c] = _uniform(rng, -0.5, 0.5, B)
                st[:, 2 + c] = sgn * _uniform(rng, 0.5, 2.0, B)
                st[:, 6], st[:, 7] = 1.2, 0.8
                act[:] = _f32(rng.uniform(-5, 5, (B, A)))
                E.append(Edge(f"wrap{c + 1}_{lab}", "cross", c, st, tm, act, lambda o, c=c, s=sgn: s * o["state"][:, c] < 0,
                              lo=np.full(B, sgn * (p.theta_max - 0.2)), hi=np.full(B, sgn * p.theta_max), K=64))
        st, tm, act = _mk(BS, F, A)
        st[:, 0] = _uniform(rng, -0.02, 0.02, BS)
        st[:, 1] = _uniform(rng, -0.02, 0.02, BS)
        st[:, 2] = _uniform(rng, -0.03, 0.03, BS)
        st[:, 3] = _uniform(rng, -0.03, 0.03, BS)
        act[:] = _f32(rng.uniform(-0.02, 0.02, (BS, A)))
        ang = rng.uniform(0, 2 * np.pi, BS)
        st[:, 7] = endy + 0.008 * np.sin(ang)
        E.append(Edge("success", "cross", 6, st, tm, act, flag_is(3), lo=np.full(BS, endx), hi=np.full(BS, endx + 0.05), K=KS))
    elif name in UGVO_NAMES:
        E += _ugvo_edges(name, p, rng)
    elif name in UGV_NAMES:
        F, A = 5, 2
        tx, ty = p.target_x, p.target_y
        bid = bool(p.bidirectional)
        box = [("x_hi", 0, p.map_x), ("x_lo", 0, 0.0), ("y_hi", 1, p.map_y), ("y_lo", 1, 0.0)]
        for lab, c, thr in box:
            s = np.array([tx, ty, 0, 0.3, 0]); s[c] = thr
            E.append(Edge(lab, "parked", c, s[None], np.zeros(1), np.zeros((1, A)), flag_is(1), center=np.array([thr])))
            E.append(Edge(lab + "+time", "priority", c, s[None], np.array([p.time_max - p.dt]), np.zeros((1, A)), flag_is(2),
                          center=np.array([thr]), cover=False))
        for lab, thr in (("phi_hi", np.pi), ("phi_lo", -np.pi)):
            s = np.array([1.0, 1.0, 0, thr, 0])
            E.append(Edge(lab, "parked", 3, s[None], np.zeros(1), np.zeros((1, A)), lambda o, t=thr: o["state"][:, 3] * t < 0,
                          center=np.array([thr])))
        s = np.array([tx - 0.05, ty, 0, 0.3, 0])
        E.append(Edge("success_parked", "parked", 0, s[None], np.zeros(1), np.zeros((1, A)), flag_is(3), center=np.array([tx - 0.05])))
        sd = np.array([[tx - 0.03, ty - 0.04, 0, 1.0, 0], [tx + 0.04, ty + 0.03, 0, -2.0, 0]])
        E.append(Edge("success_parked_diag", "parked", 1, sd, np.zeros(2), np.zeros((2, A)), flag_is(3),
                      lo=sd[:, 1] - np.sign(sd[:, 1] - ty) * 0.005, hi=sd[:, 1] + np.sign(sd[:, 1] - ty) * 0.005))
        E.append(Edge("success+time", "priority", 0, s[None], np.array([p.time_max - p.dt]), np.zeros((1, A)), flag_is(3),
                      center=np.array([tx - 0.05])))
        s = np.array([tx - 1e-4, ty, 0, 0.3, 0])   # vector_rad_oriented's `norm < 1e-4` guard: ephi (obs 2) == 0
        E.append(Edge("ephi_guard", "parked", 0, s[None], np.zeros(1), np.zeros((1, A)), lambda o: o["next_obs"][:, 2] != 0,
                      lo=np.array([tx - 2e-4]), hi=np.array([tx])))
        s = np.array([tx - 0.1, ty, 0, 0.5, 0])    # reward branch e > 0.1 (heading error 0.5 rad: u_phi = -1)
        E.append(Edge("reward_e_0.1", "parked", 0, s[None], np.zeros(1), np.zeros((1, A)), lambda o: o["reward"] < -0.5,
                      center=np.array([tx - 0.1])))
        if bid:  # sign(d) at d = 0 (heading 0: d = dx exactly) and the ephi = +-pi/2 shifts (atan2(+-dy, 0) = +-pi/2)
            for lab, dy in (("sign_d_0", 0.3), ("ephi_shift_neg", -0.3)):
                s = np.array([tx, ty - dy, 0, 0.0, 0])
                E.append(Edge(lab, "parked", 0, s[None], np.zeros(1), np.zeros((1, A)), lambda o: o["next_obs"][:, 0] > 0,
                              center=np.array([tx])))
                E.append(Edge(lab + "_ephi", "parked", 0, s[None], np.zeros(1), np.zeros((1, A)),
                              lambda o: o["next_obs"][:, 2] < 0, center=np.array([tx]), cover=False))
        E += _time_edges(name, p, np.array([1.0, 1.0, 0, 0.3, 0]), np.zeros(A), False)
        for lab, c, thr in box:
            sgn = 1 if lab.endswith("hi") else -1
            st, tm, act = _mk(B, F, A)
            st[:, 0], st[:, 1] = tx, ty
            st[:, 2] = _uniform(rng, 0.5, 2.5, B)
            st[:, 3] = (0.0 if sgn > 0 else np.pi) if c == 0 else sgn * np.pi / 2
            st[:, 3] += _uniform(rng, -0.4, 0.4, B)
            st[:, 4] = _uniform(rng, -1, 1, B)
            act[:] = _f32(rng.uniform(-3, 3, (B, A)))
            E.append(Edge(lab + "_cross", "cross", c, st, tm, act, flag_is(1), lo=np.full(B, thr - sgn * 0.2),
                          hi=np.full(B, thr + sgn * 0.01), K=64))
        for lab, sgn in (("phi_hi", 1), ("phi_lo", -1)):
            st, tm, act = _mk(B, F, A)
            st[:, 0], st[:, 1] = _uniform(rng, 1, 4, B), _uniform(rng, 1, 4, B)
            st[:, 2] = _uniform(rng, 0, 1, B)
            st[:, 4] = sgn * _uniform(rng, 0.5, 3, B)
            act[:] = _f32(rng.uniform(-3, 3, (B, A)))
            E.append(Edge(lab + "_cross", "cross", 3, st, tm, act, lambda o, s=sgn: s * o["state"][:, 3] < 0,
                          lo=np.full(B, sgn * (np.pi - 0.2)), hi=np.full(B, sgn * np.pi), K=64))
        st, tm, act = _mk(BS, F, A)
        ang = rng.uniform(0, 2 * np.pi, BS)
        st[:, 1] = ty + 0.04 * np.sin(ang)
        st[:, 2] = _uniform(rng, 0, 0.005, BS)
        st[:, 3] = _uniform(rng, -np.pi, np.pi, BS)
        st[:, 4] = _uniform(rng, -0.5, 0.5, BS)
        act[:] = _f32(rng.uniform(-0.1, 0.1, (BS, A)))
        E.append(Edge("success", "cross", 0, st, tm, act, flag_is(3), lo=np.full(BS, tx), hi=np.full(BS, tx - 0.1), K=KS))
        st, tm, act = _mk(B, F, A)
        st[:, 1] = ty
        st[:, 2] = _uniform(rng, 0.05, 0.3, B)
        st[:, 3] = _uniform(rng, 0.4, 0.8, B)
        act[:] = _f32(rng.uniform(-0.5, 0.5, (B, A)))
        E.append(Edge("reward_e_0.1_cross", "cross", 0, st, tm, act, lambda o: o["reward"] < -0.5,
                      lo=np.full(B, tx - 0.2), hi=np.full(B, tx - 0.02), K=64))
        if not bid:
            st, tm, act = _mk(B, F, A)
            st[:, 0], st[:, 1] = _uniform(rng, 1, 4, B), _uniform(rng, 1, 4, B)
            st[:, 3] = _uniform(rng, -3, 3, B)
            act[:, 0] = _f32(_uniform(rng, -3, -0.5, B))
            act[:, 1] = _f32(_uniform(rng, -3, 3, B))
            E.append(Edge("vel_clamp", "cross", 2, st, tm, act, lambda o: o["state"][:, 2] == 0,
                          lo=np.full(B, 0.1), hi=np.zeros(B), K=64))
    else:
        raise KeyError(name)
    return E


@functools.lru_cache(maxsize=None)
def lanes(name, dt=np.float64):
    """every edge lane of `name`.  dt=np.float32: the parked, priority and time lanes rebuilt for the fp32 engine (scanned
    over the floats around the float32 threshold)."""
    p = host(name)._params
    rng = np.random.default_rng(sum(map(ord, name)))
    parts, blocks, n = [], [], 0
    for e in _family_edges(name, p, rng):
        if dt == np.float32 and e.kind == "cross":
            continue
        if dt == np.float32 and e.lo is not None and e.center is None:
            sub, c, _ = _flip(name, e)
            e = Edge(**{**sub.__dict__, "center": _unord(c)})
        st, tm, act, ks = _expand(name, e, dt)
        L = len(tm)
        parts.append((st, tm, act, np.full(L, e.label, object), np.full(L, e.kind, object), ks))
        blocks.append((e, slice(n, n + L)))
        n += L
    cat = lambda i: np.concatenate([q[i] for q in parts])
    return Lanes(cat(0), cat(1), cat(2), cat(3), cat(4), cat(5), blocks)


def state_compare(name, p, a, b):
    """per-lane mixed error |a - b| / max(1, |b|) of post-step states, the wrapped angles compared modulo their period."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    d = a - b
    cols, per = ([0, 1], 2 * p.theta_max) if name == "twolink" else ([3], 2 * np.pi) if name in UGV_NAMES + UGVO_NAMES else ([], 1.0)
    d[:, cols] = (d[:, cols] + per / 2) % per - per / 2
    return np.max(np.abs(d) / np.maximum(1.0, np.abs(b)), axis=1)
