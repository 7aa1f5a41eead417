"""CPU half of the edge-lane tests (tests/env_edges.py): the lanes themselves and the oracle side of every check.

The GPU half (test_env_edges_gpu.py) holds the CUDA kernels to these lanes; what is checked here is that the lanes are
what they claim to be -- parked states do not move, every listed edge has lanes on both sides of its decision within
2 ulps, the restated reference rules agree with the C oracle -- and that the crossing lanes are fine enough to tell a
norm evaluated the reference's way from one evaluated with FMA contraction.
"""
import numpy as np
import pytest

import env_edges as E


# parked edges decided by something other than the flag (wrap, heading-error guard and shifts, reward branch)
NOT_FLAG_EDGES = ("phi_hi", "phi_lo", "ephi_guard", "reward_e_0.1", "sign_d_0", "ephi_shift_neg")

# families whose time lanes are live states (no rest state, or one that is already a success)
MOVING_TIME_LANES = ("cartpole_angleonly_ppo2", "fas", "fas_ppo2", "fas_discrete")


@pytest.fixture(scope="module", autouse=True)
def _oracle(oracle_lib):
    return oracle_lib


def _oracle_out(name, L):
    return E.oracle_step(name, L.state, L.time, L.action)


@pytest.mark.parametrize("name", E.NAMES)
def test_parked_lanes_are_bit_stationary_under_the_oracle(name):
    L = E.lanes(name)
    o = _oracle_out(name, L)
    wraps = np.isin(L.label, ["phi_hi", "phi_lo"])   # parked UGV headings beyond +-pi come back wrapped by 2 pi
    kinds = ["parked", "priority"] + ([] if name in MOVING_TIME_LANES else ["time"])
    sel = np.isin(L.kind, kinds) & ~wraps
    assert sel.sum() > 0 or name.startswith("fas"), name   # the attitude simulators have no rest state under gravity
    moved = np.any(o["state"][sel] != L.state[sel], axis=1)
    assert not moved.any(), (name, sorted(set(L.label[sel][moved])))
    if wraps.any():
        s = o["state"][wraps, 3]
        pre = L.state[wraps, 3]
        assert np.array_equal(s, np.where(pre > np.pi, pre - 2 * np.pi, np.where(pre < -np.pi, pre + 2 * np.pi, pre)))


@pytest.mark.parametrize("name", E.NAMES)
def test_oracle_flags_equal_the_restated_rule(name):
    """the restatement the GPU test holds the kernels to (env_edges.rule_flag / rule_extras) is the oracle's rule: same
    flag on every parked, time and crossing lane, and the oracle's own outputs pass every extra decision check."""
    L = E.lanes(name)
    p = E.host(name)._params
    o = _oracle_out(name, L)
    want = E.rule_flag(name, p, L.state, o["state"], o["time"])
    bad = want != o["flag"]
    assert not bad.any(), (name, sorted(set(L.label[bad])), int(bad.sum()))
    assert np.array_equal(o["done"], (o["flag"] != 0).astype(np.uint8))
    for what, m in E.rule_extras(name, p, o).items():
        assert not m.any(), (name, what, sorted(set(L.label[m])))


@pytest.mark.parametrize("name", E.NAMES)
def test_every_edge_has_lanes_on_both_sides(name):
    """coverage: every listed edge keeps lanes on both sides of its decision within 2 ulps of the flip, the time-out lanes
    put the post-step time on time_max and +-1, +-2 ulps of it, and the sub-stepped families flip between 10 and 11
    sub-steps.  Also for the float32 lanes of the fp32 engine."""
    L = E.lanes(name)
    p = E.host(name)._params
    o = _oracle_out(name, L)
    lost = []
    for e, sl in L.blocks:
        if not e.cover:
            continue
        near = np.abs(L.k[sl]) <= 2
        d = e.pred({k: v[sl] for k, v in o.items()})[near]
        if not (d.any() and (~d).any()):
            lost.append(e.label)
    assert not lost, (name, lost)
    want_labels = {e.label for e, _ in L.blocks}
    assert "time_max" in want_labels
    if name in E.SUBSTEP_NAMES:
        sub = [sl for e, sl in L.blocks if e.label == "substeps"]
        assert sub and set(o["substeps"][sub[0]]) == {10, 11}, name
    tsl = [sl for e, sl in L.blocks if e.label == "time_max"][0]
    dist = E._ord(o["time"][tsl]) - E._ord(np.float64(p.time_max))
    assert set(range(-2, 3)) <= set(dist.tolist()), (name, sorted(set(dist.tolist()) & set(range(-5, 6))))
    # float32 lanes: the fp32 rule (thresholds rounded to float32) flips within 2 float ulps on every parked edge
    L32 = E.lanes(name, np.float32)
    o32 = E.oracle_step(name, L32.state, L32.time, L32.action)
    f32 = E.rule_flag(name, p, L32.state, L32.state, o32["time"], np.float32)
    lost32 = []
    for e, sl in L32.blocks:
        if not e.cover or e.coord == E.TIME or e.label in NOT_FLAG_EDGES:
            continue
        near = np.abs(L32.k[sl]) <= 2
        if len(set(f32[sl][near].tolist())) < 2:
            lost32.append(e.label)
    assert not lost32, (name, lost32)
    # the fp32 engine's time lanes are the same float64 scan: post-step time on time_max and +-1, +-2 ulps of it
    tsl = [sl for e, sl in L32.blocks if e.label == "time_max"][0]
    dist = E._ord(o32["time"][tsl]) - E._ord(np.float64(p.time_max))
    assert set(range(-2, 3)) <= set(dist.tolist()), (name, "fp32 lanes")


@pytest.mark.parametrize("name,label", E.NORM_EDGES)
def test_norm_edges_tell_contracted_evaluation_apart(name, label):
    """sensitivity: on the oracle's post-states of the crossing lanes of every norm-based success edge, the reference
    evaluation and the other one (FMA-contracted sum of squares for CartPole, plain a*a + b*b for np.linalg.norm),
    both computed exactly, decide differently in at least one lane -- so the GPU test sees a contracted decision."""
    L = E.lanes(name)
    p = E.host(name)._params
    sl = [s for e, s in L.blocks if e.label == label and e.kind == "cross"][0]
    o = E.oracle_step(name, L.state[sl], L.time[sl], L.action[sl])
    ref = E.reference_success(name, p, o["state"])
    alt = E.contracted_success(name, p, o["state"])
    assert ref.any() and (~ref).any()
    assert (ref != alt).sum() >= 1, (name, label)


def test_ulp_helpers_walk_adjacent_doubles():
    x = np.array([-1.5, -0.0, 0.0, 5e-324, 1e-2, 3.0])
    for k in (-3, -1, 1, 2):
        y = E.ulps(x, k)
        z = x.copy()
        for _ in range(abs(k)):
            z = np.nextafter(z, np.inf if k > 0 else -np.inf)
        assert np.array_equal(y, z) or np.array_equal(np.abs(y), np.abs(z)), (k, y, z)
    f = np.array([1e-2], np.float32)
    assert E.ulps(f, 1, np.float32)[0] == np.nextafter(f[0], np.float32(1))
    a, b, c = np.array([1 + 2 ** -30]), np.array([1 - 2 ** -30]), np.array([-1.0])
    assert E.fma_exact(a, b, c)[0] == -(2.0 ** -60)
