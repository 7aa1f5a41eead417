"""GPU: K-EPISODE (csrc/episodes.cu, episodes.EpisodeTracker) against a numpy float64 restatement, and its use in
VecPPO2 (episode statistics of every rollout, vectorised deterministic evaluation).

The restatement walks t in ascending order with element-wise float64 adds across the N columns -- the same add order per
column as the kernel -- so per-instance carries and records compare bit for bit.  The statistics are sums over episodes
in another order: counts and the flag histogram are exact, every sum is within count * 2^-53 * sum|x| of the sum of the
restatement's values in extended precision (np.longdouble: 2^-64 per add, far inside the bound)."""
import math
import os
import socket
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ULP_SUM = 2.0 ** -53


def restate(r, done, flag, acc_r, acc_l, ep_r, ep_l, ep_f, first_only=False):
    """float64 loop over t; returns the final carry and records and the emitted episodes (returns, lengths, flags)."""
    acc, ln = acc_r.copy(), acc_l.astype(np.int64)
    ep_r, ep_l, ep_f = ep_r.copy(), ep_l.copy(), ep_f.copy()
    rets, lens, flags = [], [], []
    for t in range(r.shape[0]):
        acc = acc + r[t].astype(np.float64)
        ln = ln + 1
        d = done[t] != 0
        em = d & (ep_f == -1) if first_only else d
        ep_r[em], ep_l[em], ep_f[em] = acc[em], ln[em], flag[t][em]
        rets.append(acc[em])
        lens.append(ln[em])
        flags.append(flag[t][em])
        acc[d] = 0.0
        ln[d] = 0
    cat = lambda xs, dt: np.concatenate(xs).astype(dt) if xs else np.zeros(0, dt)
    return acc, ln.astype(np.int32), ep_r, ep_l, ep_f, cat(rets, np.float64), cat(lens, np.float64), cat(flags, np.int64)


def bits_equal(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def check_stats(st, rets, lens, flags):
    """stats (22 doubles) against the restatement's episodes: counts exact, sums within count * 2^-53 * sum|x|."""
    n = len(rets)
    assert st[0] == n
    hist = [int(((flags == f)).sum()) for f in range(16)] + [int(((flags < 0) | (flags > 15)).sum())]
    assert [int(v) for v in st[5:22]] == hist
    for k, x in ((1, rets), (2, rets * rets), (3, lens), (4, lens * lens)):
        exact = x.astype(np.longdouble).sum()
        assert abs(np.longdouble(st[k]) - exact) <= n * ULP_SUM * np.abs(x).astype(np.longdouble).sum(), (k, st[k], exact)


def make_inputs(T, N, pattern, r_dtype, seed):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    r = (torch.randn((T, N), generator=g, device="cuda", dtype=torch.float64) * 3.0).to(r_dtype)
    u = torch.rand((T, N), generator=g, device="cuda")
    if pattern == "none":
        done = torch.zeros((T, N), dtype=torch.bool, device="cuda")
    elif pattern == "every":
        done = torch.ones((T, N), dtype=torch.bool, device="cuda")
    elif pattern == "first":
        done = torch.zeros((T, N), dtype=torch.bool, device="cuda")
        done[0] = True
    elif pattern == "last":
        done = torch.zeros((T, N), dtype=torch.bool, device="cuda")
        done[-1] = True
    else:
        done = u < float(pattern)
    flag = torch.randint(0, 16, (T, N), generator=g, device="cuda", dtype=torch.int32)
    odd = torch.rand((T, N), generator=g, device="cuda") < 0.1          # some flags outside the histogram
    flag = torch.where(odd, torch.tensor([-3, 16, 99, 2 ** 31 - 1], device="cuda", dtype=torch.int32)[
        torch.randint(0, 4, (T, N), generator=g, device="cuda")], flag).contiguous()
    acc_r = torch.randn(N, generator=g, device="cuda", dtype=torch.float64) * 10.0   # an episode in progress
    acc_l = torch.randint(0, 50, (N,), generator=g, device="cuda", dtype=torch.int32)
    return r.contiguous(), done.to(torch.uint8).contiguous(), flag, acc_r, acc_l


def tracker_with_carry(N, acc_r, acc_l, first_only=False):
    from reinforcementlearningplatform_b200 import EpisodeTracker
    tr = EpisodeTracker(N, "cuda", first_only=first_only)
    tr.acc_return.copy_(acc_r)
    tr.acc_length.copy_(acc_l)
    return tr


def host(*ts):
    return [t.cpu().numpy() for t in ts]


def check_against_restatement(tr, r, done, flag, acc_r, acc_l, first_only=False):
    N = r.shape[-1]
    ep0 = (np.full(N, np.nan), np.full(N, -1, np.int32), np.full(N, -1, np.int32))
    rn, dn, fn, ar, al = host(r.reshape(-1, N), done.reshape(-1, N), flag.reshape(-1, N), acc_r, acc_l)
    acc, ln, ep_r, ep_l, ep_f, rets, lens, flags = restate(rn, dn, fn, ar, al, *ep0, first_only=first_only)
    g_acc, g_ln, g_r, g_l, g_f, st = host(tr.acc_return, tr.acc_length, tr.ep_return, tr.ep_length, tr.ep_flag, tr.stats)
    assert bits_equal(g_acc, acc) and bits_equal(g_ln, ln), "carry"
    assert bits_equal(g_r, ep_r) and bits_equal(g_l, ep_l) and bits_equal(g_f, ep_f), "records"
    check_stats(st, rets, lens, flags)
    return rets


# ------------------------------------------------------------------ 1. restatement sweep
SHAPES = [(T, N) for T in (1, 7, 64, 1000) for N in (1, 127, 128, 129, 100003)]
PATTERNS = ["none", "every", "first", "last", "0.01", "0.3"]


@pytest.mark.parametrize("T,N", SHAPES)
def test_scan_matches_float64_restatement(T, N):
    import torch
    for pattern in PATTERNS:
        for r_dtype in (torch.float32, torch.float64):
            r, done, flag, acc_r, acc_l = make_inputs(T, N, pattern, r_dtype, seed=T * 7919 + N)
            tr = tracker_with_carry(N, acc_r, acc_l)
            tr.update(r, done, flag)
            rets = check_against_restatement(tr, r, done, flag, acc_r, acc_l)
            if pattern == "every":      # the last episode is one step long, or the carried one plus a step if T = 1
                assert len(rets) == T * N and bool((tr.ep_length == (acc_l + 1 if T == 1 else 1)).all())
            if pattern == "none":
                assert len(rets) == 0 and bool((tr.acc_length == acc_l + T).all())


def test_one_step_buffers_and_bool_done():
    """[N] tensors (an env's own reward / is_terminal / terminal_flag after one step), done given as bool"""
    import torch
    r, done, flag, acc_r, acc_l = make_inputs(1, 5000, "0.3", torch.float32, seed=3)
    tr = tracker_with_carry(5000, acc_r, acc_l)
    tr.update(r[0], done[0].bool(), flag[0])
    check_against_restatement(tr, r, done, flag, acc_r, acc_l)


# ------------------------------------------------------------------ 2. split invariance, 3. repeatability
@pytest.mark.parametrize("N", [129, 100003])
def test_split_calls_equal_one_call(N):
    import torch
    T = 64
    r, done, flag, acc_r, acc_l = make_inputs(T, N, "0.3", torch.float32, seed=N)
    whole = tracker_with_carry(N, acc_r, acc_l)
    whole.update(r, done, flag)
    for cut in (1, T // 2, T - 1):
        part = tracker_with_carry(N, acc_r, acc_l)
        part.update(r[:cut].contiguous(), done[:cut].contiguous(), flag[:cut].contiguous())
        part.update(r[cut:].contiguous(), done[cut:].contiguous(), flag[cut:].contiguous())
        for k in ("acc_return", "acc_length", "ep_return", "ep_length", "ep_flag"):
            assert bits_equal(*host(getattr(part, k), getattr(whole, k))), (cut, k)
        sp, sw = host(part.stats, whole.stats)
        assert np.array_equal(sp[[0] + list(range(5, 22))], sw[[0] + list(range(5, 22))]), cut
        assert sw[0] > 0


def test_statistics_are_bit_reproducible():
    import torch
    T, N = 64, 100003
    r, done, flag, acc_r, acc_l = make_inputs(T, N, "0.01", torch.float32, seed=17)
    runs = []
    for _ in range(4):
        tr = tracker_with_carry(N, acc_r, acc_l)
        tr.update(r, done, flag)
        tr.update(r, done, flag)
        runs.append(tr.stats.clone())
    for s in runs[1:]:
        assert bits_equal(*host(s, runs[0]))


# ------------------------------------------------------------------ 4. first_only
@pytest.mark.parametrize("pattern", ["0.01", "0.3", "every"])
def test_first_only_records_the_first_episode(pattern):
    import torch
    T, N = 64, 10007
    r, done, flag, acc_r, acc_l = make_inputs(T, N, pattern, torch.float64, seed=5)
    tr = tracker_with_carry(N, acc_r, acc_l, first_only=True)
    cut = 20
    tr.update(r[:cut].contiguous(), done[:cut].contiguous(), flag[:cut].contiguous())
    tr.update(r[cut:].contiguous(), done[cut:].contiguous(), flag[cut:].contiguous())
    rets = check_against_restatement(tr, r, done, flag, acc_r, acc_l, first_only=True)
    never = ~done.bool().any(0)
    assert len(rets) == int((~never).sum()) <= N
    assert bool((tr.ep_flag[never] == -1).all()) and bool((tr.ep_flag[~never] != -1).all())
    # the first done row of each instance is the recorded one
    first_t = torch.argmax(done.to(torch.int32), 0)
    got = torch.gather(flag, 0, first_t.view(1, -1))[0]
    assert torch.equal(tr.ep_flag[~never], got[~never])
    if pattern == "0.01":
        assert bool(never.any())


# ------------------------------------------------------------------ 5. per-step scans == whole-rollout scan
@pytest.mark.parametrize("name", ["cartpole_angleonly_ppo2", "soi", "uav_pos"])
def test_per_step_scans_equal_rollout_scan(name):
    import torch
    from helpers import env_specs
    from reinforcementlearningplatform_b200 import EpisodeTracker, RolloutBuffer
    cls, kw = env_specs()[name]
    n, T, seed = 3000, 200, 4
    mk = lambda: cls(n_envs=n, device="cuda", dtype=torch.float64, io_dtype=torch.float32, seed=seed, auto_reset=True, **kw)
    e1, e2 = mk(), mk()
    e1.reset(True)
    e2.reset(True)
    buf = RolloutBuffer(T, e2)
    ar = torch.as_tensor(np.asarray(e1.action_range, dtype=np.float64), device="cuda", dtype=torch.float32)
    g = torch.Generator(device="cuda").manual_seed(seed)
    buf.a.copy_(ar[:, :1].view(1, -1, 1) + (ar[:, 1:] - ar[:, :1]).view(1, -1, 1) *
                torch.rand(buf.a.shape, generator=g, device="cuda"))
    t1, t2 = EpisodeTracker(n, "cuda"), EpisodeTracker(n, "cuda")
    for t in range(T):
        e1.step_soa(buf.a[t].contiguous())
        t1.update(e1.reward, e1.is_terminal, e1.terminal_flag)
    buf.collect(e2)
    t2.update(buf.r, buf.done, buf.flag)
    for k in ("acc_return", "acc_length", "ep_return", "ep_length", "ep_flag"):
        assert bits_equal(*host(getattr(t1, k), getattr(t2, k))), (name, k)
    # the statistics are summed per call, i.e. in another order: both equal the restatement within its bound
    zero_r, zero_l = torch.zeros(n, dtype=torch.float64, device="cuda"), torch.zeros(n, dtype=torch.int32, device="cuda")
    for tr in (t1, t2):
        check_against_restatement(tr, buf.r, buf.done, buf.flag, zero_r, zero_l)
    if name == "cartpole_angleonly_ppo2":
        assert t2.summary()["episodes"] > 0


# ------------------------------------------------------------------ 6. tracking inside VecPPO2
def _agent(track, reward_norm=True, n=2048, T=32, seed=5, env_seed=3):
    import torch
    import reinforcementlearningplatform_b200 as rlp
    from reinforcementlearningplatform_b200.ppo2 import VecPPO2, reference_nets
    env = rlp.CartPoleAngleOnly(n_envs=n, variant="ppo2", io_dtype=torch.float32, auto_reset=True, seed=env_seed)
    torch.manual_seed(seed)
    actor, critic = reference_nets(env.state_dim, env.action_dim, "cuda", init_std=1.2, mean_act="identity")
    agent = VecPPO2(env, actor, critic, {"buffer_size": T, "K_epochs": 2, "mini_batch_size": 8192}, std=1.2,
                    reward_norm=reward_norm, seed=seed, track_episodes=track)
    env.reset(True)
    return agent


def _flat(agent):
    return agent.fused.params.flat.detach().clone()


def test_tracking_does_not_change_training():
    import torch
    a_on, a_off = _agent(True), _agent(False)
    assert a_off.episodes is None
    for it in range(3):
        m_on, m_off = a_on.collect(), a_off.collect()
        assert m_on == m_off
        for f in ("s", "a", "a_lp", "r", "s_", "done", "flag"):
            assert torch.equal(getattr(a_on.buffer, f), getattr(a_off.buffer, f)), (it, f)
        l_on, l_off = a_on.learn(), a_off.learn()
        assert l_on == l_off
        assert torch.equal(_flat(a_on), _flat(a_off))
    assert a_on.episodes.summary()["episodes"] > 0


def test_collect_statistics_are_over_raw_rewards_across_rollouts():
    """two collects (no learn between): the tracker equals the restatement over the concatenated raw buf.r, including
    episodes that started in the first rollout; with the reward normaliser on, the statistics are the same bits"""
    import torch
    plain, normed = _agent(True, reward_norm=False), _agent(True, reward_norm=True)
    cols = []
    for _ in range(2):
        plain.collect()
        normed.collect()
        b = plain.buffer
        cols.append((b.r.clone(), b.done.clone(), b.flag.clone()))
        assert not torch.equal(normed.buffer.r, b.r)                     # normed.buffer holds normalised rewards
    r, done, flag = (torch.cat([c[k] for c in cols]) for k in range(3))
    N = r.shape[1]
    zero_r, zero_l = torch.zeros(N, dtype=torch.float64, device="cuda"), torch.zeros(N, dtype=torch.int32, device="cuda")
    check_against_restatement(plain.episodes, r, done, flag, zero_r, zero_l)
    # episodes spanning the boundary: instances with no done in rollout 1 whose episode ended in rollout 2
    spans = (~cols[0][1].bool().any(0)) & cols[1][1].bool().any(0)
    assert int(spans.sum()) > 0
    assert bits_equal(*host(plain.episodes.stats, normed.episodes.stats))
    assert bits_equal(*host(plain.episodes.ep_return, normed.episodes.ep_return))


def test_collect_reset_zeroes_the_carry():
    agent = _agent(True, reward_norm=False, T=8)
    agent.collect()
    old = agent.episodes.acc_length.clone()
    agent.env._policy_obs_valid = False        # what set_state_buffers leaves: collect() resets the env
    agent.collect()
    running = (old > 0) & ~agent.buffer.done.bool().any(0)
    assert bool(running.any())
    assert bool((agent.episodes.acc_length[running] == 8).all())


# ------------------------------------------------------------------ 7. evaluation
def _time_limit_steps(env):
    tm = getattr(env, "time_max", None) or getattr(env, "timeMax")
    return int(math.ceil(float(tm) / float(env.dt))) + 1


def _plain_eval(agent, env, max_steps):
    import torch
    N = env.n_envs
    env.reset(True)
    acc = torch.zeros(N, dtype=torch.float64, device="cuda")
    ln = torch.zeros(N, dtype=torch.int32, device="cuda")
    ret = torch.full((N,), math.nan, dtype=torch.float64, device="cuda")
    length = torch.full((N,), -1, dtype=torch.int32, device="cuda")
    flag = torch.full((N,), -1, dtype=torch.int32, device="cuda")
    fin = torch.zeros(N, dtype=torch.bool, device="cuda")
    for _ in range(max_steps):
        a = agent.evaluate(env.policy_state.t().contiguous())
        env.step_soa(a)
        acc = acc + env.reward.double()
        ln = ln + 1
        d = env.is_terminal.clone()
        new = d & ~fin
        ret[new], length[new], flag[new] = acc[new], ln[new], env.terminal_flag[new]
        fin |= d
        acc[d] = 0.0
        ln[d] = 0
        if bool(fin.all()):
            break
    return ret, length, flag


@pytest.mark.parametrize("name", ["cartpole_angleonly_ppo2", "uav_pos"])
def test_evaluation_matches_a_plain_loop(name):
    import torch
    from helpers import env_specs
    from reinforcementlearningplatform_b200.ppo2 import VecPPO2, reference_nets
    cls, kw = env_specs()[name]
    mk = lambda n, seed: cls(n_envs=n, device="cuda", dtype=torch.float64, io_dtype=torch.float32, seed=seed,
                             auto_reset=True, **kw)
    train_env = mk(1024, 3)
    torch.manual_seed(2)
    actor, critic = reference_nets(train_env.state_dim, train_env.action_dim, "cuda", init_std=0.5)
    agent = VecPPO2(train_env, actor, critic, {"buffer_size": 8, "K_epochs": 1}, std=0.5, seed=2)
    e_eval, e_plain = mk(2048, 11), mk(2048, 11)
    limit = _time_limit_steps(e_eval)
    out = agent.evaluate_episodes(e_eval, max_steps=limit + 64)
    ret, length, flag = _plain_eval(agent, e_plain, limit + 64)
    assert bool((out["ep_flag"] != -1).all()), "every instance finishes within the time limit"
    assert int(out["ep_length"].max()) <= limit
    assert bits_equal(*host(out["ep_return"], ret))
    assert torch.equal(out["ep_length"], length) and torch.equal(out["ep_flag"], flag)
    assert out["episodes"] == 2048 and sum(out["flag_counts"]) == 2048
    r64 = ret.cpu().numpy()
    assert abs(out["mean_return"] - r64.mean()) <= 1e-12 * np.abs(r64).mean() + 1e-300
    assert abs(out["mean_length"] - length.double().mean().item()) <= 1e-12 * limit
    with pytest.raises(ValueError):
        agent.evaluate_episodes(train_env, 10)
    with pytest.raises(ValueError):
        agent.evaluate_episodes(cls(n_envs=4, device="cuda", io_dtype=torch.float32, auto_reset=False, **kw), 10)


def test_evaluation_leaves_training_unchanged():
    import torch
    import reinforcementlearningplatform_b200 as rlp
    a, b = _agent(True), _agent(True)
    ev_env = rlp.CartPoleAngleOnly(n_envs=1000, variant="ppo2", io_dtype=torch.float32, auto_reset=True, seed=9)
    for it in range(2):
        a.collect()
        b.collect()
        a.learn()
        b.learn()
        steps = a.policy.step
        ms = a.reward_norm._run.clone()
        out = a.evaluate_episodes(ev_env, max_steps=300)
        assert out["episodes"] == 1000
        assert a.policy.step == steps and torch.equal(a.reward_norm._run, ms)
    a.collect()
    b.collect()
    for f in ("s", "a", "a_lp", "r", "done", "flag"):
        assert torch.equal(getattr(a.buffer, f), getattr(b.buffer, f)), f
    a.learn()
    b.learn()
    assert torch.equal(_flat(a), _flat(b))
    assert torch.equal(a.fused.exp_avg, b.fused.exp_avg) and torch.equal(a.fused.exp_avg_sq, b.fused.exp_avg_sq)
    assert bits_equal(*host(a.episodes.stats, b.episodes.stats))


# ------------------------------------------------------------------ 8. learning shows in the episode statistics
def test_example_learning_raises_episode_return_and_length():
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "examples"))
    import train_ppo2_vec as T
    log = T.main(["--env", "cartpole_angleonly", "--envs", "4096", "--steps", "64", "--iters", "25", "--epochs", "6",
                  "--eval-envs", "2048"])
    rows, ev = log[:-1], log[-1]["eval"]
    assert all(r["episodes"] > 0 for r in rows)
    for k in ("mean_episode_return", "mean_episode_length"):
        first, last = np.mean([r[k] for r in rows[:3]]), np.mean([r[k] for r in rows[-3:]])
        assert last > first, (k, first, last)
    assert all(len(r["flag_counts"]) == 17 and sum(r["flag_counts"]) == r["episodes"] for r in rows)
    assert ev["episodes"] == 2048 and np.isfinite(ev["mean_return"])


# ------------------------------------------------------------------ 9. two ranks on one device
N_TOTAL, T_DIST, SEED_DIST = 2049, 300, 3


def _dist_actions():
    import torch
    g = torch.Generator().manual_seed(21)
    return (torch.rand((T_DIST, 1, N_TOTAL), generator=g) * 10.0 - 5.0).to(torch.float32)   # CartPoleAngleOnly: [-5, 5]


def _run_tracker(n, off, group=None):
    import torch
    import reinforcementlearningplatform_b200 as rlp
    env = rlp.CartPoleAngleOnly(n_envs=n, variant="ppo2", io_dtype=torch.float32, auto_reset=True, seed=SEED_DIST,
                                env_index_offset=off)
    env.reset(True)
    acts = _dist_actions()[:, :, off:off + n].cuda()
    tr = rlp.EpisodeTracker(n, "cuda", group=group)
    rows = []
    for t in range(T_DIST):
        env.step_soa(acts[t].contiguous())
        tr.update(env.reward, env.is_terminal, env.terminal_flag)
        rows.append((env.reward.clone(), env._done.clone(), env.terminal_flag.clone()))
    return tr, rows


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK="0")
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(0)
    dist.init_process_group("gloo")
    from reinforcementlearningplatform_b200 import dist as D
    n, off = D.shard(N_TOTAL, rank, world)
    tr, _ = _run_tracker(n, off)
    q.put((rank, n, off, tr.summary()))
    dist.destroy_process_group()


def test_two_ranks_sum_to_one_tracker():
    import torch
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=300) for _ in procs)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    (_, n0, o0, s0), (_, n1, o1, s1) = res
    assert (n0, o0, n1, o1) == (1025, 0, 1024, 1025)
    tr, rows = _run_tracker(N_TOTAL, 0)
    one = tr.summary()
    r, done, flag = (torch.stack([x[k] for x in rows]) for k in range(3))
    z = np.zeros(N_TOTAL)
    _, _, _, _, _, rets, lens, flags = restate(*host(r, done, flag), z, z.astype(np.int32), z, z.astype(np.int32),
                                               np.full(N_TOTAL, -1, np.int32))
    n = len(rets)
    assert n >= N_TOTAL and one["episodes"] == n
    for s in (s0, s1):
        assert s["episodes"] == one["episodes"] and s["flag_counts"] == one["flag_counts"]
        for k, x in (("mean_return", rets), ("mean_length", lens)):
            exact = float(x.astype(np.longdouble).sum()) / n
            bound = (n + 2) * ULP_SUM * float(np.abs(x).astype(np.longdouble).sum()) / n
            assert abs(s[k] - exact) <= bound and abs(one[k] - exact) <= bound, (k, s[k], one[k], exact)
        for k in ("std_return", "std_length"):
            assert math.isclose(s[k], one[k], rel_tol=1e-9), (k, s[k], one[k])
