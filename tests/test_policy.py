"""Batched policy forward (csrc/policy.cu) against vectors recorded from the reference's own PPOActor_Gaussian /
PPOCritic (utils/classes.py:529-623) and choose_action (Proximal_Policy_Optimization2.py:69-76).  float32: the kernel
sums in k order, torch in GEMM blocks, so the bar is 2e-6 absolute on mean / value (stated here), and the derived
action / log-prob follow with the same budget scaled by 1 / std^2."""
import os

import numpy as np
import pytest

from helpers import GOLDEN


def cases():
    with np.load(os.path.join(GOLDEN, "policy.npz")) as z:
        g = {k: z[k] for k in z.files}
    return [{k[len(f"c{i}_"):]: v for k, v in g.items() if k.startswith(f"c{i}_")} for i in range(int(g["n_cases"]))]


def numpy_forward(c):
    """float64 restatement of the two nets (the CPU-side checker of the fixtures themselves)."""
    h = c["s"].astype(np.float64)
    for l in ("fc1", "fc2", "fc3"):
        h = np.tanh(h @ c[f"actor_{l}_w"].astype(np.float64).T + c[f"actor_{l}_b"])
    mean = np.maximum(h @ c["actor_mean_layer_w"].astype(np.float64).T + c["actor_mean_layer_b"], 0.0)
    v = c["s"].astype(np.float64)
    for l in ("fc1", "fc2"):
        v = np.tanh(v @ c[f"critic_{l}_w"].astype(np.float64).T + c[f"critic_{l}_b"])
    v = v @ c["critic_fc3_w"].astype(np.float64).T + c["critic_fc3_b"]
    return mean, v[:, 0]


def test_fixture_is_consistent_with_a_float64_restatement():
    for c in cases():
        mean, v = numpy_forward(c)
        np.testing.assert_allclose(c["mean"], mean, atol=2e-6)
        np.testing.assert_allclose(c["value"], v, atol=2e-6)
        std = float(c["std"])
        a = np.clip(mean + std * c["eps"], c["a_min"], c["a_max"])
        np.testing.assert_allclose(c["action"], a, atol=3e-6)
        lp = -((c["action"].astype(np.float64) - mean) ** 2) / (2 * std * std) - np.log(std) - 0.5 * np.log(2 * np.pi)
        np.testing.assert_allclose(c["log_prob"], lp, atol=2e-5)


def _build(c, torch):
    def lin(w, b):
        l = torch.nn.Linear(w.shape[1], w.shape[0])
        with torch.no_grad():
            l.weight.copy_(torch.from_numpy(w))
            l.bias.copy_(torch.from_numpy(b))
        return l.cuda()
    actor = [lin(c[f"actor_{n}_w"], c[f"actor_{n}_b"]) for n in ("fc1", "fc2", "fc3", "mean_layer")]
    critic = [lin(c[f"critic_{n}_w"], c[f"critic_{n}_b"]) for n in ("fc1", "fc2", "fc3")]
    return actor, critic


@pytest.mark.gpu
@pytest.mark.parametrize("precision,tol", [("fp32", 2e-6), ("umma", 5e-6)])
def test_engine_policy_matches_reference_nets(precision, tol):
    import torch
    import reinforcementlearningplatform_b200 as rlp
    for c in cases():
        actor, critic = _build(c, torch)
        pol = rlp.GaussianPolicy(actor, critic, c["a_min"], c["a_max"], float(c["std"]), precision=precision)
        obs = torch.from_numpy(np.ascontiguousarray(c["s"].T)).cuda()
        eps = torch.from_numpy(np.ascontiguousarray(c["eps"].T)).cuda()
        out = pol(obs, noise=eps, want_mean=True)
        f = lambda t: t.cpu().numpy().T
        np.testing.assert_allclose(f(out["mean"]), c["mean"], atol=tol)
        np.testing.assert_allclose(out["value"].cpu().numpy(), c["value"], atol=tol)
        np.testing.assert_allclose(f(out["action"]), c["action"], atol=tol + 1e-6)
        np.testing.assert_allclose(f(out["log_prob"]), c["log_prob"], atol=10 * tol)
        lo, hi = c["a_min"][None, :], c["a_max"][None, :]
        assert np.all(f(out["action"]) >= lo) and np.all(f(out["action"]) <= hi)
        # critic-only and actor-only calls give the same numbers
        v2 = rlp.GaussianPolicy(None, critic, c["a_min"], c["a_max"], 1.0, precision=precision)(obs)["value"]
        assert torch.equal(v2, out["value"])
        a2 = rlp.GaussianPolicy(actor, None, c["a_min"], c["a_max"], float(c["std"]), precision=precision)(obs, noise=eps)["action"]
        assert torch.equal(a2, out["action"])


@pytest.mark.gpu
def test_engine_policy_sampling_statistics_and_determinism():
    """In-kernel Philox + Box-Muller draws: N(0, 1) moments over 1 M x 8 samples, independent of sharding and of the
    launch, different per step."""
    import torch
    import reinforcementlearningplatform_b200 as rlp
    c = cases()[0]
    actor, critic = _build(c, torch)
    n = 1 << 20
    obs = torch.zeros(6, n, dtype=torch.float32, device="cuda")
    wide = (np.full(8, -1e9, np.float32), np.full(8, 1e9, np.float32))
    pol = rlp.GaussianPolicy(actor, critic, *wide, 0.5, seed=11)
    o = pol(obs, want_mean=True)
    z = ((o["action"] - o["mean"]) / 0.5).double()
    assert abs(float(z.mean())) < 5e-3 and abs(float(z.std()) - 1.0) < 5e-3
    assert abs(float((z ** 3).mean())) < 2e-2 and abs(float((z ** 4).mean()) - 3.0) < 5e-2
    assert abs(float(torch.corrcoef(z[:2])[0, 1])) < 5e-3          # the two Box-Muller outputs are uncorrelated
    o2 = pol(obs)                                                  # next step: fresh draws
    assert not torch.equal(o2["action"], o["action"])
    # the same (seed, global index, step) gives the same draw whatever the shard
    half = rlp.GaussianPolicy(actor, critic, *wide, 0.5, seed=11, env_index_offset=n // 2)
    oh = half(obs[:, n // 2:].contiguous())
    assert torch.equal(oh["action"], o["action"][:, n // 2:])


@pytest.mark.gpu
def test_policy_drives_env_on_device():
    """policy_state -> K-POLICY -> action -> step kernel with float32 I/O, all on the engine's own buffers."""
    import torch
    import reinforcementlearningplatform_b200 as rlp
    c = cases()[0]
    actor, critic = _build(c, torch)
    n = 4096
    env = rlp.UavPosCtrlRL(n_envs=n, random_trajectory=True, auto_reset=True, io_dtype=torch.float32, seed=1)
    env.reset(True)
    pol = rlp.GaussianPolicy(actor, critic, c["a_min"], c["a_max"], float(c["std"]), seed=2)
    for t in range(10):
        out = pol(env._reset_obs)
        env.step_soa(out["action"])
    assert torch.isfinite(env.reward).all() and float(env.time.max()) == pytest.approx(0.2)
    assert out["value"].shape == (n,) and out["log_prob"].shape == (8, n)


def wide_case():
    with np.load(os.path.join(GOLDEN, "policy_wide.npz")) as z:
        return {k: z[k] for k in z.files}


def test_wide_fixture_is_consistent_with_a_float64_restatement():
    c = wide_case()
    h = c["s"].astype(np.float64)
    for l in ("fc1", "fc2"):
        h = np.tanh(h @ c[f"actor_{l}_w"].astype(np.float64).T + c[f"actor_{l}_b"])
    off = (c["a_min"].astype(np.float64) + c["a_max"]) / 2
    mean = np.tanh(h @ c["actor_mean_layer_w"].astype(np.float64).T + c["actor_mean_layer_b"]) * (c["a_max"] - off) + off
    v = c["s"].astype(np.float64)
    for k in range(2):
        v = np.tanh(v @ c[f"critic_l{k}_w"].astype(np.float64).T + c[f"critic_l{k}_b"])
    v = (v @ c["critic_l2_w"].astype(np.float64).T + c["critic_l2_b"])[:, 0]
    np.testing.assert_allclose(c["mean"], mean, atol=2e-5)
    np.testing.assert_allclose(c["value"], v, atol=2e-5)


@pytest.mark.gpu
def test_engine_policy_matches_the_256_wide_dppo2_demo_nets():
    """41-256-256-2 actor with the tanh range head and per-dimension std, 41-256-256-1 critic
    (demonstration/DPPO2/DPPO2-4-UGVForwardObstacleAvoidance/train.py:26-107): weights streamed through shared memory.
    Tolerance 2e-5 absolute on mean / value: 256-term float32 sums (the reference's own float32 GEMM is ~1e-5 from the
    float64 restatement above), head gain up to 2 pi."""
    import torch
    import reinforcementlearningplatform_b200 as rlp
    c = wide_case()

    def lin(w, b):
        l = torch.nn.Linear(w.shape[1], w.shape[0])
        with torch.no_grad():
            l.weight.copy_(torch.from_numpy(w))
            l.bias.copy_(torch.from_numpy(b))
        return l.cuda()
    actor = [lin(c[f"actor_{n}_w"], c[f"actor_{n}_b"]) for n in ("fc1", "fc2", "mean_layer")]
    critic = [lin(c[f"critic_l{k}_w"], c[f"critic_l{k}_b"]) for k in range(3)]
    pol = rlp.GaussianPolicy(actor, critic, c["a_min"], c["a_max"], c["std"], actor_out_act="tanh_range")
    # 400 fixture rows, tiled to cover several 128-instance tiles per CTA and a ragged last tile
    reps = 53
    obs = torch.from_numpy(np.ascontiguousarray(np.tile(c["s"], (reps, 1)).T)).cuda()
    eps = torch.from_numpy(np.ascontiguousarray(np.tile(c["eps"], (reps, 1)).T)).cuda()
    out = pol(obs, noise=eps, want_mean=True)
    f = lambda t: t.cpu().numpy().T
    tol = 2e-5
    for name, t in (("mean", tol), ("action", tol + 1e-6), ("log_prob", 10 * tol)):
        np.testing.assert_allclose(f(out[name]), np.tile(c[name], (reps, 1)), atol=t, err_msg=name)
    np.testing.assert_allclose(out["value"].cpu().numpy(), np.tile(c["value"], reps), atol=tol)
    with pytest.raises(ValueError):
        rlp.GaussianPolicy(actor, critic, c["a_min"], c["a_max"], c["std"], precision="fp32")  # vector std: umma only


@pytest.mark.gpu
def test_umma_policy_sees_optimizer_steps_and_ragged_sizes():
    """the packed weight copy follows in-place parameter updates; n need not be a multiple of the 128-instance tile.
    Rows: the reference nets (policy_umma16.cu) and nets with 41 observation fields, more than policy_umma16.cu holds
    (the resident modes of policy_umma.cu)."""
    import torch
    import reinforcementlearningplatform_b200 as rlp
    c = cases()[0]
    torch.manual_seed(0)
    lins = lambda dims: [torch.nn.Linear(i, o).cuda() for i, o in zip(dims[:-1], dims[1:])]
    for actor, critic in (_build(c, torch), (lins((41, 64, 64, 32, 8)), lins((41, 64, 32, 1)))):
        S = actor[0].in_features
        pol = rlp.GaussianPolicy(actor, critic, c["a_min"], c["a_max"], float(c["std"]))
        ref = rlp.GaussianPolicy(actor, critic, c["a_min"], c["a_max"], float(c["std"]), precision="fp32")
        for n in (1, 127, 129, 1000, 128 * 148 * 2 + 77):
            obs = torch.randn(S, n, device="cuda")
            eps = torch.randn(8, n, device="cuda")
            a, b = pol(obs, noise=eps, want_mean=True), ref(obs, noise=eps, want_mean=True)
            for k in ("mean", "action", "value"):
                assert float((a[k] - b[k]).abs().max()) <= 7e-6, (S, n, k)
        with torch.no_grad():
            for l in actor + critic:
                l.weight.mul_(0.5)
                l.bias.add_(0.1)
        obs = torch.randn(S, 777, device="cuda")
        eps = torch.randn(8, 777, device="cuda")
        a, b = pol(obs, noise=eps, want_mean=True), ref(obs, noise=eps, want_mean=True)
        assert float((a["mean"] - b["mean"]).abs().max()) <= 7e-6 and float((a["value"] - b["value"]).abs().max()) <= 7e-6


def test_wide_nets_are_rejected_by_the_fp32_kernel_not_silently_slow():
    """nets that do not fit the shared-memory design of policy.cu return B200ENV_ESIZE there (the tcgen05 kernel streams
    them; no fallback path exists); any precision other than B200_POLICY_FP32 (0) returns B200ENV_EPARAMS"""
    import ctypes as C
    from reinforcementlearningplatform_b200 import _lib
    lib = _lib.load()
    m = _lib.MLP()
    m.n_layers = 3
    for i, d in enumerate((41, 256, 256, 2)):
        m.dims[i] = d
    for l in range(3):
        m.w[l] = 1 << 20
        m.b[l] = 1 << 20
    m.out_act = 1
    for precision, want in ((0, -6), (1, -3)):
        rc = lib.b200_policy_forward(16, C.byref(m), None, C.c_void_p(1 << 20), C.c_void_p(1 << 20), C.c_void_p(1 << 20),
                                     C.c_float(0.5), None, 0, 0, 0, precision, C.c_void_p(1 << 20), None, None, None, None)
        assert rc == want, precision
    import reinforcementlearningplatform_b200 as rlp
    with pytest.raises(ValueError):
        rlp.GaussianPolicy(None, None, [0.0], [1.0], 1.0, precision="fp16")
