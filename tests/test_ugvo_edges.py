"""CPU half of the UGV-FOA lanes of tests/ugvo_edges.py: the lanes are what they claim to be under the C oracle."""
import numpy as np
import pytest

import env_edges as E
import ugvo_edges as U
from helpers import ENGINE_TOL


@pytest.fixture(scope="module", autouse=True)
def _oracle(oracle_lib):
    return oracle_lib


@pytest.mark.parametrize("name", E.UGVO_NAMES)
def test_tie_lanes_are_parked_and_the_tie_decides_rays(name):
    """the tied circles sit at bit-equal centre distance, the lanes do not move under a zero action, no lane collides,
    and exchanging the two circles moves rays of every lane by more than 1000 x ENGINE_TOL (the GPU test's bound): the
    lower-index rule is visible in the laser."""
    p = E.host(name)._params
    rows = U.tie_rows(p)
    d = [E.np_norm2(rows[:, 0] - rows[:, 8 + 3 * k], rows[:, 1] - rows[:, 9 + 3 * k]) for k in (0, 1)]
    assert np.array_equal(d[0], d[1])
    o = E.oracle_step(name, rows, np.zeros(len(rows)), np.zeros((len(rows), 2)))
    assert np.array_equal(o["state"], rows) and not (o["flag"] == 4).any()
    a, b = U.oracle_observe(name, rows), U.oracle_observe(name, U.swap_first_two(rows))
    assert np.array_equal(a, o["obs"]) and np.array_equal(a, o["next_obs"])
    tol = ENGINE_TOL[name]
    gap = np.max(np.abs(a[:, 4:] - b[:, 4:]) / np.maximum(1.0, np.abs(b[:, 4:])), axis=1)
    assert (gap > 1e3 * tol).all(), (int((gap <= 1e3 * tol).sum()), float(gap.min()))


@pytest.mark.parametrize("name", E.UGVO_NAMES)
def test_map_edges_reach_their_fallbacks(name):
    """under the oracle: `target_fallback` keeps block 64's target (restated from the Philox draws) and places no circle;
    the give-up envs stop short of obs_num in some instances and zero the slots after n_obs; `full_16` fills all 16."""
    p0 = E.host(name)._params
    n = 64
    for label, over in U.MAP_EDGES.items():
        p = U.with_params(p0, over)
        st, _ = U.oracle_reset(name, n, p)
        nobs = st[:, 7].astype(int)
        want = min(p.obs_num, 16)
        for i in range(n):
            assert not st[i, 8 + 3 * nobs[i]:].any(), (label, i)
        if label == "target_fallback":
            assert (nobs == 0).all()
            lo, hx, hy = p.st_margin, p.map_x - p.st_margin, p.map_y - p.st_margin
            for i in range(n):
                u0, u1 = U.draw2(E.SEED, i, 0, 64)
                assert (st[i, 5], st[i, 6]) == (U.lerp_u(lo, hx, u0), U.lerp_u(lo, hy, u1)), i
                u0, u1 = U.draw2(E.SEED, i, 0, 0)
                assert (st[i, 0], st[i, 1]) == (U.lerp_u(lo, hx, u0), U.lerp_u(lo, hy, u1)), i
        elif label.startswith("give_up"):
            assert (nobs < want).all() and (nobs > 0).all(), (label, np.bincount(nobs))
        else:
            assert (nobs == want).all(), (label, np.bincount(nobs))


@pytest.mark.parametrize("name", E.UGVO_NAMES)
def test_fake_laser_restatement_equals_the_oracle(name):
    """ugvo_edges.fake_laser (numpy float64, the reference's expressions) equals observe() of the C oracle bit for bit on
    every laser block, the tie lanes, the pose-level edge lanes and 4096 freshly reset maps."""
    p = E.host(name)._params
    o = U.oracle_env(name, 4096)
    o.reset()
    parts = [rows for rows, _, _ in U.laser_blocks(p).values()] + [U.tie_rows(p), o.state.T.copy()]
    L = E.lanes(name)
    parts.append(L.state[np.isin(L.kind, ["parked", "priority", "time"])])
    rows = np.concatenate(parts)
    got = U.laser_obs(p, U.fake_laser(p, rows))
    want = U.oracle_observe(name, rows)[:, 4:]
    bad = np.any(got != want, axis=1)
    assert not bad.any(), (int(bad.sum()), len(rows))


@pytest.mark.parametrize("name", E.UGVO_NAMES)
def test_laser_blocks_sit_on_their_decisions(name):
    """every laser block: its sensitive rays (the restated value moves by more than the one-step bound over the
    perturbation set P) are a minority, and among its stable rays both outcomes of its decision occur -- two values
    apart by more than 1e3 x the bound on one ray over the scan, or, where both outcomes give the same range (in-range
    boundary and segment end, the circle on the normal, ray length at laser_dis), both sides of the decisive test."""
    from test_engine_gpu import ONE_STEP_TOL
    p = E.host(name)._params
    tol = ONE_STEP_TOL[name]
    for lab, (rows, ks, _) in U.laser_blocks(p).items():
        base, V = U.laser_variants(p, rows)
        ob, ov = U.laser_obs(p, base), U.laser_obs(p, V)
        sens = np.any(np.abs(ov - ob) > tol, axis=0)
        assert sens.sum() < 0.5 * sens.size, (lab, int(sens.sum()), sens.size)
        both = np.nanmax(np.where(sens, np.nan, ob), axis=0) - np.nanmin(np.where(sens, np.nan, ob), axis=0)
        sides = U.block_decision(p, lab, rows)
        assert np.nanmax(both) > 1e3 * tol or (sides is not None and sides.any() and (~sides).any()), lab


@pytest.mark.parametrize("name", E.UGVO_NAMES)
def test_equality_cases_decide_both_ways(name):
    """the reset's legality tests at equality under the oracle: obstacle 0 is the restated first candidate exactly
    when fl(r + safety_dis_st) lies below its distance from the start (k < 0), and the target is the first candidate
    exactly when safety_dis_st <= its distance (k <= 0)."""
    p = E.host(name)._params
    cases = U.equality_cases(p)
    assert {lab for lab, *_ in cases} == {"start", "target"}
    for lab, gid, over, k in cases:
        st, _ = U.oracle_reset(name, 1, U.with_params(p, over), offset=gid)
        if lab == "start":
            a, b, c = U.draw3(E.SEED, gid, 0, 1000)
            first = st[0, 8] == U.lerp_u(0., p.map_x, a) and st[0, 9] == U.lerp_u(0., p.map_y, b)
            assert first == (k < 0), (lab, gid, k)
        else:
            u0, u1 = U.draw2(E.SEED, gid, 0, 1)
            first = st[0, 5] == U.lerp_u(p.st_margin, p.map_x - p.st_margin, u0)
            assert first == (k <= 0), (lab, gid, k)
