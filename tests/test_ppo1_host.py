"""CPU: the argument checks of the PPO v1 entries (b200_mc_returns_stats, b200_ppo1_grad) return their error codes before
any CUDA call, VecPPO's defaults, and VecPPO2.set_action_std's shape rule."""
import ctypes as C
import inspect
import types

import pytest


@pytest.fixture(scope="module")
def lib():
    import os
    import __graft_entry__ as g
    from reinforcementlearningplatform_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        g.build()
    return _lib.load()


ESIZE, EDTYPE, ENULL, EPARAMS = -6, -2, -4, -3
P = C.c_void_p(0x1000)        # never dereferenced: every call below fails its checks first
BIG = C.c_void_p(0x10000)


def ret_stats(lib, r_dtype=1, T=4, N=300, r=P, done=P, ret=P, stats=P, scratch=BIG, scratch_bytes=1 << 20):
    return lib.b200_mc_returns_stats(r_dtype, T, N, r, done, 0.99, ret, stats, scratch, scratch_bytes, None)


def test_mc_returns_stats_error_codes(lib):
    for T, N in ((0, 5), (-1, 5), (5, 0), (5, -3), (5, 1 << 31), (5, 1 << 40)):
        assert ret_stats(lib, T=T, N=N) == ESIZE, (T, N)
    for dt in (-1, 2, 7):
        assert ret_stats(lib, r_dtype=dt) == EDTYPE
    for k in ("r", "done", "ret", "stats", "scratch"):
        assert ret_stats(lib, **{k: None}) == ENULL, k
    # scratch: K-GAE's per-block partials, b200_gae_scratch_bytes(N) bytes, 8-byte aligned
    need = lib.b200_gae_scratch_bytes(300)
    assert need > 0
    assert ret_stats(lib, scratch_bytes=need - 8) == EPARAMS
    assert ret_stats(lib, scratch=C.c_void_p(0x10004)) == EPARAMS
    # precedence: size before dtype before null before params
    assert ret_stats(lib, T=0, r_dtype=9, r=None) == ESIZE
    assert ret_stats(lib, r_dtype=9, r=None, scratch_bytes=0) == EDTYPE
    assert ret_stats(lib, r=None, scratch_bytes=0) == ENULL


def _mlp(dims, out_act=0):
    from reinforcementlearningplatform_b200 import _lib
    m = _lib.MLP()
    m.n_layers = len(dims) - 1
    for l, d in enumerate(dims):
        m.dims[l] = d
    for l in range(m.n_layers):
        m.w[l], m.b[l] = 0x2000 + 0x100 * l, 0x3000 + 0x100 * l
    m.out_act = out_act
    return m


def _batch(**kw):
    from reinforcementlearningplatform_b200 import _lib
    b = _lib.PPO2Batch()
    b.T, b.N = 4, 300
    b.s, b.a, b.a_lp, b.adv, b.v_target = (k << 20 for k in range(1, 6))   # 1 MB apart: no two ranges overlap
    b.index, b.first, b.count, b.perm_key = None, 0, 1200, 0
    for k, v in kw.items():
        setattr(b, k, v)
    return b


def ppo1(lib, batch=None, actor=None, critic=None, std=0.5, a_min=P, a_max=P, value_coef=0.5, value=None, ga=P, gc=P,
         loss=P, ws=BIG, ws_bytes=None, no_actor=False, no_critic=False, no_batch=False):
    am = actor or _mlp((6, 64, 64, 32, 8), 1)
    cm = critic or _mlp((6, 64, 32, 1))
    if ws_bytes is None:
        ws_bytes = lib.b200_ppo2_workspace_bytes(C.byref(am), C.byref(cm))
    b = batch or _batch()
    return lib.b200_ppo1_grad(None if no_batch else C.byref(b), None if no_actor else C.byref(am),
                              None if no_critic else C.byref(cm), std, None, a_min, a_max, 0.2, 0.01, value_coef, value,
                              ga, gc, loss, ws, ws_bytes, None)


def test_ppo1_grad_error_codes(lib):
    # both nets and the batch are required
    assert ppo1(lib, no_batch=True) == ENULL
    assert ppo1(lib, no_actor=True) == ENULL
    assert ppo1(lib, no_critic=True) == ENULL
    # value_coef < 0 or NaN
    for vc in (-0.5, -1e-30, float("nan")):
        assert ppo1(lib, value_coef=vc) == EPARAMS, vc
    # pointers b200_ppo2_grad needs; adv is the output of the advantage launch, v_target holds R_hat
    for field in ("s", "a", "a_lp", "adv", "v_target"):
        assert ppo1(lib, batch=_batch(**{field: None})) == ENULL, field
    for k in ("ga", "gc", "loss", "ws"):
        assert ppo1(lib, **{k: None}) == ENULL, k
    assert ppo1(lib, actor=_mlp((6, 64, 2), 2), a_min=None) == ENULL    # the tanh-range head reads a_min / a_max
    # parameters
    assert ppo1(lib, std=0.0) == EPARAMS
    assert ppo1(lib, actor=_mlp((6, 64, 8), 3)) == EPARAMS               # unknown head
    assert ppo1(lib, critic=_mlp((6, 64, 2))) == EPARAMS                 # critic output != 1
    assert ppo1(lib, critic=_mlp((5, 64, 1))) == EPARAMS                 # state_dim mismatch
    # sizes
    for kw in (dict(T=0), dict(N=0), dict(N=1 << 31), dict(count=0), dict(first=-1), dict(first=1, count=1200)):
        assert ppo1(lib, batch=_batch(**kw)) == ESIZE, kw
    assert ppo1(lib, actor=_mlp((6, 128, 8), 1)) == ESIZE                # wider than 64
    assert ppo1(lib, ws_bytes=1024) == ESIZE                              # workspace too small
    # precedence: the required nets before value_coef before the rest
    assert ppo1(lib, no_critic=True, value_coef=-1.0) == ENULL
    assert ppo1(lib, value_coef=-1.0, batch=_batch(T=0)) == EPARAMS


def test_vecppo_defaults():
    from reinforcementlearningplatform_b200 import VecPPO, VecPPO2, ppo, ppo2
    m = ppo.DEFAULT_PPO1_MSG
    assert m["set_adam_eps"] is False and m["use_grad_clip"] is False and m["use_lr_decay"] is False
    assert m["value_coef"] == 0.5 and m["ret_norm_eps"] == 1e-7
    # the keys VecPPO shares with VecPPO2 keep VecPPO2's values
    for k in ("entropy_coef", "eps_clip", "gamma", "K_epochs", "a_lr", "c_lr", "buffer_size"):
        assert m[k] == ppo2.DEFAULT_PPO_MSG[k], k
    assert (m["entropy_coef"], m["eps_clip"], m["gamma"]) == (0.01, 0.2, 0.99)
    assert issubclass(VecPPO, VecPPO2)
    sig = inspect.signature(VecPPO.__init__).parameters
    assert sig["reward_norm"].default is False and "learner" not in sig
    assert inspect.signature(VecPPO2.__init__).parameters["reward_norm"].default is True   # VecPPO2 unchanged
    assert ppo2.DEFAULT_PPO_MSG["set_adam_eps"] is True and ppo2.DEFAULT_PPO_MSG["use_grad_clip"] is True


def _holder(std):
    import torch
    t = torch.as_tensor(std, dtype=torch.float32).reshape(-1)
    vec = t.clone() if t.numel() > 1 else None
    part = lambda: types.SimpleNamespace(std=float(t[0]) if vec is None else 1.0, std_vec=None if vec is None else vec.clone())
    return types.SimpleNamespace(std=t.clone(), policy=part(), fused=part())


def test_set_action_std_keeps_the_form_of_std():
    from reinforcementlearningplatform_b200 import VecPPO2
    scalar = _holder(0.5)
    for bad in ([0.3, 0.3], [[0.3]], [0.2, 0.3, 0.4]):
        with pytest.raises(ValueError):
            VecPPO2.set_action_std(scalar, bad)
    for bad in (0.0, -0.3, float("nan"), float("inf")):
        with pytest.raises(ValueError):
            VecPPO2.set_action_std(scalar, bad)
    assert float(scalar.std[0]) == 0.5 and scalar.policy.std == 0.5 and scalar.fused.std == 0.5   # untouched
    VecPPO2.set_action_std(scalar, 0.3)
    import numpy as np
    f = float(np.float32(0.3))
    assert float(scalar.std[0]) == f and scalar.policy.std == f and scalar.fused.std == f
    vector = _holder([0.4, 0.5, 0.6])
    for bad in (0.3, [0.3, 0.3], [0.1, 0.2, 0.3, 0.4], [[0.1, 0.2, 0.3]]):
        with pytest.raises(ValueError):
            VecPPO2.set_action_std(vector, bad)
    VecPPO2.set_action_std(vector, [0.1, 0.2, 0.3])
    for t in (vector.std, vector.policy.std_vec, vector.fused.std_vec):
        assert t.tolist() == np.float32([0.1, 0.2, 0.3]).tolist()


def test_ppo1_grad_rejects_outputs_that_overlap_inputs(lib):
    """adv and value are written by the advantage launch while R_hat (v_target), s, a, a_lp and the index are read: an
    overlap is B200ENV_EPARAMS before any CUDA call (T = 4, N = 300: a [T][N] column is 4800 bytes)"""
    b0 = _batch()
    col = 4 * 300 * 4
    assert ppo1(lib, batch=_batch(adv=b0.v_target)) == EPARAMS                       # the in-place call
    assert ppo1(lib, batch=_batch(adv=b0.v_target + col - 4)) == EPARAMS             # partial overlap
    assert ppo1(lib, batch=_batch(adv=b0.s + 6 * col - 4)) == EPARAMS                # last element of s [T][6][N]
    assert ppo1(lib, batch=_batch(adv=b0.a + 8 * col - 4)) == EPARAMS                # a [T][8][N]
    assert ppo1(lib, batch=_batch(adv=b0.a_lp)) == EPARAMS
    idx = 6 << 20
    assert ppo1(lib, batch=_batch(index=idx, first=10, count=100, adv=idx + 8 * 109)) == EPARAMS
    for v in (b0.adv, b0.v_target, b0.adv + col - 4, b0.s):
        assert ppo1(lib, value=C.c_void_p(v)) == EPARAMS, hex(v)
