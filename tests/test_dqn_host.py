"""CPU: K-DQN's C entries return their error codes before any CUDA call, the replay sampler evaluated on the host
(b200_dqn_sample_indices) stays inside the valid window and is uniform, and VecDQN checks its arguments on a host-only
env."""
import ctypes as C

import numpy as np
import pytest
import torch


@pytest.fixture(scope="module")
def lib():
    import os
    import __graft_entry__ as g
    from reinforcementlearningplatform_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        g.build()
    return _lib.load()


ESIZE, ENULL, EPARAMS = -6, -4, -3
P = C.c_void_p(0x1000)        # never dereferenced: every call below fails its checks first


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


NET = (2, 64, 64, 47)
N = 300


def act(lib, n=N, q=None, obs=1 << 20, table=2 << 20, eps=0.1, index=3 << 20, value=4 << 20, q_out=None, no_q=False):
    m = q or _mlp(NET)
    v = lambda x: None if x is None else C.c_void_p(x)
    return lib.b200_dqn_act(n, None if no_q else C.byref(m), v(obs), v(table), eps, 1, 2, 0, v(index), v(value), v(q_out),
                            None)


def test_act_error_codes(lib):
    for k in ("obs", "table", "index", "value"):
        assert act(lib, **{k: None}) == ENULL, k
    assert act(lib, no_q=True) == ENULL
    m = _mlp(NET)
    m.w[1] = 0
    assert act(lib, q=m) == ENULL
    for n in (0, -1, 1 << 31):
        assert act(lib, n=n) == ESIZE, n
    for dims in ((2, 65, 47), (65, 64, 47), (2, 64, 65)):
        assert act(lib, q=_mlp(dims)) == ESIZE, dims
    five = _mlp((2, 8, 8, 8, 47))
    five.n_layers = 5
    assert act(lib, q=five) == ESIZE
    for eps in (-0.01, 1.01, float("nan"), float("inf")):
        assert act(lib, eps=eps) == EPARAMS, eps
    assert act(lib, q=_mlp(NET, out_act=1)) == EPARAMS
    # outputs overlapping inputs or each other
    assert act(lib, index=(1 << 20) + 4 * 17) == EPARAMS                      # inside obs [2][N]
    assert act(lib, value=(2 << 20) + 8) == EPARAMS                           # inside table [47]
    assert act(lib, value=(3 << 20) + 4 * (N - 1)) == EPARAMS                 # last element of index
    assert act(lib, q_out=(5 << 20), value=(5 << 20) + 4 * 46 * N) == EPARAMS  # inside q_out [47][N]
    assert act(lib, index=0x2000 + 64) == EPARAMS                             # a weight of the net
    # precedence: null before size before params
    assert act(lib, n=0, obs=None, eps=2.0) == ENULL
    assert act(lib, n=0, eps=2.0) == ESIZE


def _batch(**kw):
    from reinforcementlearningplatform_b200 import _lib
    b = _lib.DQNBatch()
    b.R, b.N = 16, N
    b.s, b.r, b.s_, b.a, b.done = (k << 20 for k in range(1, 6))            # 1 MB apart: no two ranges overlap
    b.newest_row, b.valid_rows, b.count, b.index, b.sample_key = 3, 15, 1000, None, 7
    for k, v in kw.items():
        setattr(b, k, v)
    return b


def grad(lib, batch=None, q=None, qt=None, gamma=0.99, g=8 << 20, loss=9 << 20, ws=10 << 20, ws_bytes=None,
         no_batch=False, no_q=False, no_qt=False):
    m, mt = q or _mlp(NET), qt or _mlp(NET)
    for l in range(mt.n_layers):
        mt.w[l], mt.b[l] = 0x6000 + 0x100 * l, 0x7000 + 0x100 * l
    b = batch or _batch()
    if ws_bytes is None:
        ws_bytes = lib.b200_dqn_workspace_bytes(C.byref(m), b.count)
    v = lambda x: None if x is None else C.c_void_p(x)
    return lib.b200_dqn_grad(None if no_batch else C.byref(b), None if no_q else C.byref(m),
                             None if no_qt else C.byref(mt), gamma, 1, v(g), v(loss), v(ws), ws_bytes, None)


def test_workspace_bytes(lib):
    m = _mlp(NET)
    need = lib.b200_dqn_workspace_bytes(C.byref(m), 4096)
    assert need >= 4096 * 4 + (64 * 2 + 64 + 64 * 64 + 64 + 47 * 64 + 47) * 4
    assert lib.b200_dqn_workspace_bytes(C.byref(m), 0) == 0
    assert lib.b200_dqn_workspace_bytes(C.byref(_mlp((2, 64, 65))), 4096) == 0
    assert lib.b200_dqn_workspace_bytes(None, 4096) == 0


def test_grad_error_codes(lib):
    for k in ("no_batch", "no_q", "no_qt"):
        assert grad(lib, **{k: True}) == ENULL, k
    for k in ("g", "loss", "ws"):
        assert grad(lib, **{k: None}) == ENULL, k
    for k in ("s", "r", "s_", "a", "done"):
        assert grad(lib, batch=_batch(**{k: None})) == ENULL, k
    for kw in (dict(R=1, valid_rows=0, newest_row=0), dict(N=0), dict(N=1 << 31), dict(R=1 << 31), dict(count=0),
               dict(count=-5)):
        assert grad(lib, batch=_batch(**kw), ws_bytes=1 << 30) == ESIZE, kw
    assert grad(lib, q=_mlp((2, 64, 65)), ws_bytes=1 << 30) == ESIZE
    assert grad(lib, q=_mlp((65, 64, 47)), qt=_mlp((65, 64, 47)), ws_bytes=1 << 30) == ESIZE
    need = lib.b200_dqn_workspace_bytes(C.byref(_mlp(NET)), 1000)
    assert grad(lib, ws_bytes=need - 4) == ESIZE
    assert grad(lib, gamma=float("nan")) == EPARAMS
    for kw in (dict(valid_rows=0), dict(valid_rows=16), dict(valid_rows=-1), dict(newest_row=-1), dict(newest_row=16)):
        assert grad(lib, batch=_batch(**kw)) == EPARAMS, kw
    assert grad(lib, qt=_mlp((2, 64, 32, 47))) == EPARAMS                     # shapes differ
    assert grad(lib, q=_mlp(NET, out_act=1), qt=_mlp(NET, out_act=1)) == EPARAMS
    # outputs overlapping inputs, weights or each other
    assert grad(lib, g=(1 << 20) + 64) == EPARAMS                             # inside s
    assert grad(lib, loss=(4 << 20) + 4 * N) == EPARAMS                       # inside a
    assert grad(lib, g=(5 << 20)) == EPARAMS                                  # done
    assert grad(lib, ws=0x6000 - 64) == EPARAMS                               # workspace over the target's weights
    assert grad(lib, loss=0x2000 + 4) == EPARAMS                              # the online net's weight
    assert grad(lib, loss=(8 << 20) + 16) == EPARAMS                          # inside grad
    assert grad(lib, batch=_batch(index=(9 << 20) - 64)) == EPARAMS           # index [1000] int64 under loss_out
    # precedence: null before size before params
    assert grad(lib, batch=_batch(count=0, valid_rows=0), loss=None) == ENULL
    assert grad(lib, batch=_batch(count=0, valid_rows=0), ws_bytes=1 << 30) == ESIZE


def sample(lib, key, newest, V, R, n, first, count):
    out = (C.c_int64 * max(count, 1))()
    rc = lib.b200_dqn_sample_indices(key, newest, V, R, n, first, count, out)
    assert rc == 0
    return np.frombuffer(out, dtype=np.int64, count=count).copy()


def restated_sampler(key, j, newest, V, R, n):
    """The sampler of csrc/learn.cu, restated: splitmix64 of key + (j + 1) * golden, multiply-high onto [0, V N)."""
    from reinforcementlearningplatform_b200.dqn import _mix
    b = (_mix(key, j) * (V * n)) >> 64
    return ((newest - b // n) % R) * n + b % n


def test_sample_indices_errors(lib):
    out = (C.c_int64 * 4)()
    assert lib.b200_dqn_sample_indices(1, 0, 1, 1, 8, 0, 4, out) == ESIZE
    assert lib.b200_dqn_sample_indices(1, 0, 1, 4, 0, 0, 4, out) == ESIZE
    assert lib.b200_dqn_sample_indices(1, 0, 1, 4, 8, -1, 4, out) == ESIZE
    assert lib.b200_dqn_sample_indices(1, 0, 1, 4, 8, 0, -1, out) == ESIZE
    assert lib.b200_dqn_sample_indices(1, 0, 4, 4, 8, 0, 4, out) == EPARAMS
    assert lib.b200_dqn_sample_indices(1, 0, 0, 4, 8, 0, 4, out) == EPARAMS
    assert lib.b200_dqn_sample_indices(1, 4, 3, 4, 8, 0, 4, out) == EPARAMS
    assert lib.b200_dqn_sample_indices(1, 0, 3, 4, 8, 0, 4, None) == ENULL
    assert lib.b200_dqn_sample_indices(1, 0, 3, 4, 8, 0, 0, None) == 0


@pytest.mark.parametrize("R,n,k", [(8, 100, 3), (8, 100, 8), (8, 100, 21), (64, 7, 1000), (5, 1 << 20, 2)])
def test_sample_indices_window(lib, R, n, k):
    """After k collection steps the valid rows are the min(k, R - 1) newest ones; the in-flight row k % R never appears."""
    V, newest = min(k, R - 1), (k - 1) % R
    p = sample(lib, 0xC0FFEE + k, newest, V, R, n, 0, 20000)
    rows, inst = p // n, p % n
    valid = {(newest - b) % R for b in range(V)}
    assert set(np.unique(rows).tolist()) <= valid
    assert not np.any(rows == k % R) or V == 0
    assert inst.min() >= 0 and inst.max() < n
    # bit for bit the restated statement, at a few positions including a far `first`
    for j in (0, 1, 777, 19999):
        assert p[j] == restated_sampler(0xC0FFEE + k, j, newest, V, R, n)
    far = sample(lib, 0xC0FFEE + k, newest, V, R, n, (1 << 40) + 5, 3)
    assert far.tolist() == [restated_sampler(0xC0FFEE + k, (1 << 40) + 5 + j, newest, V, R, n) for j in range(3)]


def test_sample_indices_keys(lib):
    a = sample(lib, 2 ** 64 - 3, 5, 7, 8, 1000, 0, 4096)
    assert np.array_equal(a, sample(lib, 2 ** 64 - 3, 5, 7, 8, 1000, 0, 4096))
    assert np.array_equal(a[100:200], sample(lib, 2 ** 64 - 3, 5, 7, 8, 1000, 100, 100))   # position-only
    b = sample(lib, 2 ** 64 - 2, 5, 7, 8, 1000, 0, 4096)
    assert np.mean(a == b) < 0.01


def test_sample_indices_uniform(lib):
    """Chi-square of the counts over the V valid rows and over the N instances of 2^20 draws."""
    from scipy.stats import chi2
    R, n, V, newest = 16, 97, 11, 2
    p = sample(lib, 12345, newest, V, R, n, 0, 1 << 20)
    back = (newest - p // n) % R
    for counts, cells in ((np.bincount(back, minlength=V), V), (np.bincount(p % n, minlength=n), n),
                          (np.bincount(back * n + p % n, minlength=V * n), V * n)):
        assert counts.size == cells
        e = p.size / cells
        stat = float(((counts - e) ** 2 / e).sum())
        assert chi2.sf(stat, cells - 1) > 1e-4, (cells, stat)


# ------------------------------------------------------------------------------------------------ VecDQN arguments
def _env(**kw):
    import reinforcementlearningplatform_b200 as rlp
    kw.setdefault("io_dtype", torch.float32)
    return rlp.FlightAttitudeSimulatorDiscrete(n_envs=8, host_only=True, **kw)


def test_vecdqn_argument_checks(lib):
    import reinforcementlearningplatform_b200 as rlp
    from reinforcementlearningplatform_b200 import _lib
    from reinforcementlearningplatform_b200.dqn import q_net
    env = _env()
    A = env.action_num[0]
    assert A == 46 and env.state_dim == 2 and env.action_dim == 1   # int((3.0 + 1.6) / 0.1 + 1): 46.99.. truncates
    net = q_net(env.state_dim, A, "cpu")
    cont = rlp.Flight_Attitude_Simulator(n_envs=8, host_only=True, io_dtype=torch.float32)
    with pytest.raises(ValueError, match="discrete"):
        rlp.VecDQN(cont, net)
    with pytest.raises(ValueError, match="float32"):
        rlp.VecDQN(_env(io_dtype=torch.float64, dtype=torch.float64), net)
    with pytest.raises(ValueError, match="unknown"):
        rlp.VecDQN(env, net, {"memory_size": 10})
    for msg in ({"memory_capacity": 1}, {"batch_size": 0}, {"target_replace_iter": 0}, {"learn_start": 0},
                {"gamma": float("nan")}):
        with pytest.raises(ValueError):
            rlp.VecDQN(env, net, msg)
    for eps in (-0.1, 1.5, float("nan")):
        with pytest.raises(ValueError, match="epsilon"):
            rlp.VecDQN(env, net, epsilon=eps)
    with pytest.raises(_lib.B200EnvError, match="K-DQN"):
        rlp.VecDQN(env, q_net(env.state_dim, A, "cpu", hidden=(128,)))
    with pytest.raises(_lib.B200EnvError, match="K-DQN"):
        rlp.VecDQN(env, q_net(env.state_dim, A, "cpu", hidden=(8, 8, 8, 8)))
    with pytest.raises(ValueError, match="maps"):
        rlp.VecDQN(env, q_net(env.state_dim, 16, "cpu"))
    with pytest.raises(ValueError, match="maps"):
        rlp.VecDQN(env, q_net(3, A, "cpu"))
    # every argument right: the host-only mirror has no device, and there is no CPU path
    w0 = net[0].weight.data_ptr()
    with pytest.raises(_lib.B200EnvError, match="CPU path"):
        rlp.VecDQN(env, net)
    assert net[0].weight.data_ptr() == w0          # nothing was moved before the checks failed


def test_restated_key_schedule():
    """Sampling keys depend on the seed and the update counter only."""
    from reinforcementlearningplatform_b200.dqn import _mix
    assert _mix(5, 0) != _mix(5, 1) != _mix(6, 0)
    assert 0 <= _mix(2 ** 64 - 1, 2 ** 40) < 2 ** 64
