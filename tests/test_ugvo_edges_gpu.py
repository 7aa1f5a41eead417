"""GPU: K-UGVO (csrc/ugvo.cu) on the lanes of tests/ugvo_edges.py and on the identities between its launch paths.

  ties            two circles at bit-equal centre distance: the step's scan A (`obs`) and scan B (`next_obs`), built by
                  the per-thread insertion sort, and b200env_observe, built by the warp-vote rank, all equal the oracle
                  (lower index first).
  obs reuse       the same actions over several auto-resetting steps with `reuse_obs` on (the previous step's policy
                  observation, partly written by the warp path, stands in for scan A) and off: the same bits.
  work list       the autoreset kernel's ticket list and its `done`-scan branch reset the same instances the same way.
  neighbours      permuting the lanes of a batch permutes the outputs, bit for bit (the step kernel shares its shared
                  memory among 64 instances).
  sizes           batches of 1, 63, 64, 65 and 4097 write the bits of the same lanes inside a larger batch.
  map fallbacks   reset(random=True) with the target fallback, placement giving up and 16 circles: every state field
                  equals the oracle's bit for bit.
  equality        the reset's legality tests with fl(r + safety_dis_st) or safety_dis_st on the decisive distance.
  laser blocks    the slope error K measured; every ray of the blocks against the float64 restatement over the
                  perturbation set P (fp64), and float32 I/O rounding the fp64 values once.
"""
import numpy as np
import pytest

import env_edges as E
import ugvo_edges as U
from helpers import ENGINE_TOL, env_specs

pytestmark = pytest.mark.gpu

OUTS = ("obs", "next_obs", "reset_obs", "reward", "done", "flag", "state", "time", "episode")


def _env(name, n, auto_reset=False, offset=0, reuse_obs=None, io_dtype=None, params=None):
    import torch
    cls, kw = env_specs()[name]
    env = cls(n_envs=n, device="cuda", dtype=torch.float64, io_dtype=io_dtype, seed=E.SEED, auto_reset=auto_reset,
              env_index_offset=offset, reuse_obs=reuse_obs, **kw)
    if params:
        for k, v in params.items():
            setattr(env._params, k, v)
    return env


def _inject(env, state, time, episode=None):
    import torch
    env.set_state_buffers(torch.from_numpy(np.ascontiguousarray(np.asarray(state, np.float64).T)),
                          torch.from_numpy(np.asarray(time, np.float64)),
                          torch.from_numpy(np.zeros(len(time), np.int32) if episode is None else np.asarray(episode, np.int32)))


def _outs(env):
    import torch
    torch.cuda.synchronize()
    f = lambda x: np.ascontiguousarray(x.detach().cpu().numpy().T)
    return dict(obs=f(env._obs), next_obs=f(env._next_obs), reset_obs=f(env._reset_obs), reward=f(env._reward),
                done=f(env._done), flag=f(env._flag), state=f(env._state), time=f(env._time), episode=f(env._episode))


def _step(env, act):
    import torch
    env.step_soa(torch.from_numpy(np.ascontiguousarray(np.asarray(act).T)).to("cuda", env.io_dtype))
    return _outs(env)


def _same(a, b, keys=OUTS, what=""):
    for k in keys:
        x, y = np.ascontiguousarray(a[k]), np.ascontiguousarray(b[k])
        bad = (x.view(np.uint8) != y.view(np.uint8)).reshape(len(x), -1).any(axis=1)
        assert not bad.any(), (what, k, int(bad.sum()), np.nonzero(bad)[0][:8].tolist())


def _random_lanes(name, n):
    """n freshly reset instances (engine-drawn maps) -> lanes-first state."""
    env = _env(name, n)
    env.reset(True)
    return _outs(env)["state"].astype(np.float64)


def _mixed_lanes(name, n_random=4096):
    """the pose-level edge lanes of env_edges, the tie lanes and n_random freshly reset instances, with their times."""
    L = E.lanes(name)
    p = E.host(name)._params
    ties = U.tie_rows(p)
    st = np.concatenate([L.state, ties, _random_lanes(name, n_random)])
    tm = np.concatenate([L.time, np.zeros(len(ties) + n_random)])
    return st, tm


def _actions(rng, n, T):
    lo, hi = np.array([-3.0, -2 * np.pi]), np.array([3.0, 2 * np.pi])
    return [rng.uniform(lo, hi, (n, 2)) for _ in range(T)]


@pytest.mark.parametrize("name", E.UGVO_NAMES)
def test_tied_circles_lower_index_first_in_every_path(name, oracle_lib):
    """scan A, scan B and b200env_observe on the tie lanes (and their slot-swapped twins) equal the oracle within the
    one-step laser bound; the two tie-breaks differ by far more than the bound on every lane (CPU test)."""
    p = E.host(name)._params
    rows = np.concatenate([U.tie_rows(p), U.swap_first_two(U.tie_rows(p))])
    n = len(rows)
    want = U.oracle_observe(name, rows)
    tol = ENGINE_TOL[name]
    env = _env(name, n)
    _inject(env, rows, np.zeros(n))
    g = _step(env, np.zeros((n, 2)))
    env2 = _env(name, n)
    _inject(env2, rows, np.zeros(n))
    env2.observe()
    g["observe"] = _outs(env2)["next_obs"]
    for k in ("obs", "next_obs", "observe"):
        err = np.max(np.abs(g[k] - want) / np.maximum(1.0, np.abs(want)), axis=1)
        assert (err <= tol).all(), (name, k, int((err > tol).sum()), float(err.max()))


@pytest.mark.parametrize("name", E.UGVO_NAMES)
def test_obs_reuse_writes_the_bits_of_recomputed_scans(name):
    """six auto-resetting steps with the same actions, `reuse_obs` on and off: every output and the state, bit for
    bit, after every step; b200env_observe at the injected poses equals the first step's scan A."""
    st, tm = _mixed_lanes(name)
    n = len(tm)
    rng = np.random.default_rng(7)
    acts = _actions(rng, n, 6)
    on, off = _env(name, n, True, reuse_obs=True), _env(name, n, True, reuse_obs=False)
    assert on.reuse_obs and not off.reuse_obs
    obs_env = _env(name, n)
    for e in (on, off, obs_env):
        _inject(e, st, tm)
    obs_env.observe()
    first = _outs(obs_env)["next_obs"]
    resets = 0
    for t, a in enumerate(acts):
        go, gf = _step(on, a), _step(off, a)
        if t == 0:
            assert np.array_equal(gf["obs"].view(np.uint8), first.view(np.uint8)), name
        _same(go, gf, what=(name, t))
        resets += int(gf["done"].sum())
    assert resets >= n // 20, (name, resets)


@pytest.mark.parametrize("name", E.UGVO_NAMES)
def test_work_list_and_done_scan_reset_alike(name):
    """one auto-resetting step where most lanes time out: the ticket-list branch of ugvo_autoreset_kernel and its
    `done`-scan branch (no work list) leave the same states, maps, reset observations and episode counters."""
    st, tm = _mixed_lanes(name)
    n = len(tm)
    rng = np.random.default_rng(8)
    tm = np.where(rng.uniform(size=n) < 0.6, E.host(name)._params.time_max - 0.01, tm)
    a = _actions(rng, n, 1)[0]
    lst, scan = _env(name, n, True), _env(name, n, True)
    scan._work = None
    for e in (lst, scan):
        _inject(e, st, tm)
    gl, gs = _step(lst, a), _step(scan, a)
    assert gl["done"].sum() >= n // 2, (name, int(gl["done"].sum()), n)
    assert (gl["episode"] > 0).sum() == gl["done"].sum()
    _same(gl, gs, what=name)


@pytest.mark.parametrize("name", E.UGVO_NAMES)
def test_lane_permutation_permutes_the_outputs(name):
    """auto-reset off (a reset is keyed by the global instance index): a permuted batch gives the permuted outputs."""
    st, tm = _mixed_lanes(name)
    n = len(tm)
    rng = np.random.default_rng(9)
    a = _actions(rng, n, 1)[0]
    perm = rng.permutation(n)
    e1, e2 = _env(name, n), _env(name, n)
    _inject(e1, st, tm)
    _inject(e2, st[perm], tm[perm])
    g1, g2 = _step(e1, a), _step(e2, a[perm])
    _same({k: v[perm] for k, v in g1.items()}, g2, what=name)


@pytest.mark.parametrize("n", [1, 63, 64, 65, 4097])
@pytest.mark.parametrize("name", E.UGVO_NAMES)
def test_batch_size_does_not_change_a_lane(name, n):
    """n lanes taken from position 37 of an 8192-lane batch, with env_index_offset = 37 so that their auto-resets draw
    the same maps: three steps write the same bits as inside the large batch (partial 64-instance step blocks, partial
    4-warp aux blocks, partial 32-lane reset groups)."""
    st, tm = _mixed_lanes(name, 8192)
    rng = np.random.default_rng(10)
    sel = rng.choice(len(tm), 8192, replace=False)
    st, tm = st[sel], tm[sel]
    N, at = len(tm), 37
    acts = _actions(rng, N, 3)
    big, small = _env(name, N, True), _env(name, n, True, offset=at)
    _inject(big, st, tm)
    _inject(small, st[at:at + n], tm[at:at + n])
    for t, a in enumerate(acts):
        gb, gs = _step(big, a), _step(small, a[at:at + n])
        _same({k: v[at:at + n] for k, v in gb.items()}, gs, what=(name, n, t))


@pytest.mark.parametrize("label", sorted(U.MAP_EDGES))
@pytest.mark.parametrize("name", E.UGVO_NAMES)
def test_map_fallbacks_equal_the_oracle(name, label, oracle_lib):
    """reset(random=True) under the parameters of MAP_EDGES[label], 4096 instances at an offset across 2^32: every
    state field (start, target, heading, n_obs, every circle slot) equal to the oracle's bit for bit, and the reset
    observation within the one-step bound."""
    n, off = 4096, 2 ** 32 - 1000
    env = _env(name, n, offset=off, params=U.MAP_EDGES[label])
    env.reset(True)
    g = _outs(env)
    st, nx = U.oracle_reset(name, n, env._params, offset=off)
    _same(g, dict(state=st), keys=("state",), what=(name, label))
    assert (g["episode"] == 1).all()
    err = np.max(np.abs(g["next_obs"] - nx) / np.maximum(1.0, np.abs(nx)), axis=1)
    assert (err <= ENGINE_TOL[name]).all(), (name, label, float(err.max()))


def _laser_engine(name, rows, io_dtype=None):
    """the laser terms of scan A, scan B (a parked step) and b200env_observe at the lanes -> three [lanes, rays]."""
    n = len(rows)
    env = _env(name, n, io_dtype=io_dtype)
    _inject(env, rows, np.zeros(n))
    g = _step(env, np.zeros((n, 2)))
    env2 = _env(name, n, io_dtype=io_dtype)
    _inject(env2, rows, np.zeros(n))
    env2.observe()
    return {"obs": g["obs"][:, 4:], "next_obs": g["next_obs"][:, 4:], "observe": _outs(env2)["next_obs"][:, 4:]}


def test_slope_error_is_within_k():
    """K measured: the kernel's slope is fm64::sincos's s / c through fm64::div; over every ray of the laser blocks,
    |fl(s / c) - tan(phi)| in ulps of tan(phi), plus 1 for the division, stays within K_SLOPE (|m| < 1e3) and
    K_STEEP (steeper rays)."""
    import ctypes
    import torch
    from reinforcementlearningplatform_b200 import _lib
    lib = _lib.load()
    for name in E.UGVO_NAMES:
        p = E.host(name)._params
        ph = np.concatenate([U.ray_angles(p, rows).ravel() for rows, _, _ in U.laser_blocks(p).values()])
        xd = torch.from_numpy(ph).cuda()
        s, c = torch.empty_like(xd), torch.empty_like(xd)
        _lib.check(lib.b200_fastmath_eval(0, xd.numel(), ctypes.c_void_p(xd.data_ptr()), ctypes.c_void_p(s.data_ptr()),
                                          ctypes.c_void_p(c.data_ptr()), None), "b200_fastmath_eval")
        torch.cuda.synchronize()
        m = U.c_tan(ph)
        e = np.abs(s.cpu().numpy() / c.cpu().numpy() - m) / np.spacing(np.abs(m)) + 1
        steep = np.abs(m) >= 1e3
        print(f"{name}: slope error {e[~steep].max():.2f} ulps (|m| < 1e3, {int((~steep).sum())} rays), "
              f"{e[steep].max():.2f} ulps (|m| >= 1e3, {int(steep.sum())} rays)")
        assert e[~steep].max() <= U.K_SLOPE and e[steep].max() <= U.K_STEEP, name


@pytest.mark.parametrize("name", E.UGVO_NAMES)
def test_laser_blocks_against_the_restatement(name, oracle_lib):
    """every ray of every laser block, in scan A, scan B and b200env_observe: where the restated laser gives one value
    over the perturbation set P (within the one-step bound) the engine matches it; elsewhere (the sensitive set) the
    engine is within the bound of one of the values over P, or inside their [min, max] widened by the bound.  Printed:
    per block the lanes, the sensitive rays and the restatement's decision counts."""
    from test_engine_gpu import ONE_STEP_TOL
    p = E.host(name)._params
    tol = ONE_STEP_TOL[name]
    for lab, (rows, ks, _) in U.laser_blocks(p).items():
        stats = {}
        U.fake_laser(p, rows, stats=stats)
        base, V = U.laser_variants(p, rows)
        ob, ov = U.laser_obs(p, base), U.laser_obs(p, V)
        allv = np.concatenate([ob[None], ov])
        sens = np.any(np.abs(ov - ob) > tol, axis=0)
        print(f"{name} {lab}: {len(rows)} lanes, {int(sens.sum())} of {sens.size} rays sensitive, {stats}")
        for k, g in _laser_engine(name, rows).items():
            err = np.abs(g - ob) / np.maximum(1.0, np.abs(ob))
            bad = ~sens & (err > tol)
            assert not bad.any(), (name, lab, k, "stable", int(bad.sum()), float(err[bad].max()))
            near = np.min(np.abs(allv - g[None]) / np.maximum(1.0, np.abs(allv)), axis=0) <= tol
            inside = (g >= allv.min(0) - tol) & (g <= allv.max(0) + tol)
            bad = sens & ~near & ~inside
            assert not bad.any(), (name, lab, k, "sensitive", int(bad.sum()))


@pytest.mark.parametrize("name", E.UGVO_NAMES)
def test_laser_blocks_float32_io_round_once(name):
    """float32 I/O: every laser output of the blocks is the fp64 engine's value rounded once to float32, bit for bit."""
    import torch
    p = E.host(name)._params
    rows = np.concatenate([r for r, _, _ in U.laser_blocks(p).values()])
    g64, g32 = _laser_engine(name, rows), _laser_engine(name, rows, io_dtype=torch.float32)
    for k in g64:
        assert np.array_equal(g32[k].view(np.uint32), g64[k].astype(np.float32).view(np.uint32)), (name, k)


@pytest.mark.parametrize("name", E.UGVO_NAMES)
def test_reset_legality_at_equality_equals_the_oracle(name, oracle_lib):
    """one small env per scanned value: fl(r + safety_dis_st) on the distance from the start to obstacle 0's first
    candidate (and +-1, 2 ulps), and safety_dis_st on the first target candidate's distance: every reset field equal to
    the oracle's bit for bit."""
    p = E.host(name)._params
    for lab, gid, over, k in U.equality_cases(p):
        env = _env(name, 1, offset=gid, params=over)
        env.reset(True)
        st, _ = U.oracle_reset(name, 1, env._params, offset=gid)
        _same(_outs(env), dict(state=st), keys=("state",), what=(name, lab, gid, k))
