"""VecPPO2 as a whole: every PPO2 iteration (collect() + learn()) against a float64 torch restatement of the learner the
module cites (Proximal_Policy_Optimization2.py:78-170), on one GPU and on two ranks.

The restatement (``restate_iteration``) follows the cited lines, not VecPPO2's code, and starts every iteration from an
exact re-sync of the agent: parameters, Adam state, the permutation key or torch generator, learning rates, total_steps
and the reward normaliser's ``(n, mean, S)``.  Its inputs are the rollout buffer after ``collect()`` and the raw reward
column, captured by wrapping ``reward_norm.normalize_rows`` so that it clones its input first (the only hook).  Steps:
  1. reward rows: row t enters the running statistics after rows < t, its N samples (of every rank, in rank order)
     merged as one batch each (``normalization.merge_stats_reference``), and is normalised with the statistics after row
     t (``std = mean`` while n == 1);
  2. V(s), V(s') by the float64 critic; GAE backwards with success = done and flag != TIMEOUT_FLAG; v_target = adv + V;
     ``(adv - mean) / (std_unbiased + 1e-5)`` over all ranks' samples;
  3. index sets: ``b200_ppo2_permutation(key + e, B, first, count)`` (fused) or ``torch.randperm`` from the saved
     generator state (torch learner), mini-batch j = positions ``[j mb, min((j + 1) mb, B))`` in one process, or
     ``(B_r j) // n_mb`` on every rank of a group, with the agreed ``n_mb = min_r ceil(B_r / mb)``;
  4. per mini-batch: actor loss ``-min(r A, clamp(r) A) - entropy_coef H``, mean, (the ranks' means summed and times
     1 / world), ``clip_grad_norm_(0.5)``, ``torch.optim.Adam``; then the critic's ``mse_loss``, clip and Adam;
  5. the linear learning-rate decay after the loop, on the env steps of the whole group.
Each stage of the engine is compared with it separately, so that a failure names the stage.  Bounds: ``C * 2^-24 *
scale`` with the scale models of test_policy_routes_gpu.py (values, means, log-probs) and of K-GAE (a float64 pass over
the absolute values of the scan); parameters after ``learn()`` within the 1e-6 (actor) / 2e-6 (critic) of
test_learn_gpu.py, with the float32 restatement's distance printed beside the engine's.  The measured values are printed.
Samples within 1e-4 of a clip edge or of a relu head's kink would make float32 and float64 take different branches:
the restatement counts them and every case asserts there are none."""
import copy
import ctypes as C
import math
import os
import pickle
import socket
import sys

import numpy as np
import pytest
import torch

EPS32 = 2.0 ** -24
TANH_UNITS = 8.0       # test_policy_routes_gpu.py: SFU tanh and the operand pair of the next layer, units of 2^-24
# 10x the largest value measured on a B200 (1000 W power limit) over every case and iteration below (printed by the
# tests; DESIGN 4(m)).  Units of 2^-24 scale unless stated.
C_LP = 2.0             # collect()'s log-probs and evaluate()'s clamped mean: 0.196 measured (case f)
C_VALUE = 0.7          # V(s), V(s') of the critic-only K-POLICY launches: 0.0699 (case f, 256 wide)
C_REWARD = 10.0        # normalised reward, scale |r| + 2^-29 (|x| + |mean|) / (std + 1e-8): 0.999 (two ranks)
C_GAE = 7.2            # adv / v_target of K-GAE, scale = the scan's absolute-value pass: 0.714 (case b)
# Parameters after learn(), max |p - p64|: the 1e-6 / 2e-6 of test_learn_gpu.py / test_ppo1_gpu.py.  Measured 1.06e-7
# (actor, case e) and 1.27e-7 (critic, case e); the float32 restatement is as far from float64 as the engine is, within
# 1e-8 -- the floor is float32's own rounding of parameters near 1 -- so 10x below that floor is not reachable.
PARAM_TOL = (1e-6, 2e-6)
MOMENT_TOL = 1.4e-5    # max |exp_avg - ref| / max |ref| per net, and exp_avg_sq: 1.39e-6 both (critic, case f)
LOSS_TOL = 3.1e-5      # |loss - ref| / |ref| of the last mini-batch: 3.07e-6 (actor, case d)
KINK = 1e-4
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------------------ helpers
def _lib():
    from reinforcementlearningplatform_b200 import _lib
    return _lib


def keyed_positions(key: int, B: int, first: int, count: int) -> np.ndarray:
    """samples b = t * N + i at positions [first, first + count) of K-LEARN's keyed permutation (host evaluation)"""
    L = _lib()
    out = np.empty(count, dtype=np.int64)
    L.check(L.load().b200_ppo2_permutation(int(key) & (2 ** 64 - 1), B, first, count,
                                           out.ctypes.data_as(C.POINTER(C.c_int64))), "b200_ppo2_permutation")
    return out


def mini_batch_bounds(B: int, mb: int, n_mb: int, grouped: bool = False):
    """positions of the n_mb mini-batches of one epoch: one process, BatchSampler's [j mb, min((j + 1) mb, B)); a rank of
    a group, its own B split evenly over the n_mb the group agreed on, (B j) // n_mb"""
    if grouped:
        return [(B * j) // n_mb for j in range(n_mb + 1)]
    assert n_mb == -(-B // mb)
    return [min(j * mb, B) for j in range(n_mb + 1)]


def fused_index_sets(key: int, B: int, mb: int, n_mb: int, k_epochs: int, grouped: bool = False):
    bounds = mini_batch_bounds(B, mb, n_mb, grouped)
    return [[keyed_positions(key + e, B, bounds[j], bounds[j + 1] - bounds[j]) for j in range(n_mb)]
            for e in range(k_epochs)]


def torch_index_sets(gen_state, device, B: int, mb: int, n_mb: int, k_epochs: int, grouped: bool = False):
    g = torch.Generator(device=device)
    g.set_state(gen_state)
    bounds = mini_batch_bounds(B, mb, n_mb, grouped)
    sets = []
    for _ in range(k_epochs):
        perm = torch.randperm(B, device=device, generator=g)
        sets.append([perm[bounds[j]:bounds[j + 1]] for j in range(n_mb)])
    return sets, g.get_state()


def _linears(net):
    from reinforcementlearningplatform_b200.policy import linear_layers
    return linear_layers(net)


def _flat(net):
    return torch.cat([t.detach().reshape(-1) for lin in _linears(net) for t in (lin.weight, lin.bias)])


def _load_flat(net, flat):
    o = 0
    with torch.no_grad():
        for lin in _linears(net):
            for t in (lin.weight, lin.bias):
                t.copy_(flat[o:o + t.numel()].view_as(t))
                o += t.numel()


def _layers64(net, flat):
    """[(W, b)] float64 of ``net``'s linear layers taken from the flat parameter vector"""
    out, o = [], 0
    for lin in _linears(net):
        W = flat[o:o + lin.weight.numel()].double().view_as(lin.weight)
        o += lin.weight.numel()
        b = flat[o:o + lin.bias.numel()].double()
        o += lin.bias.numel()
        out.append((W, b))
    return out


def _net64(layers, x, f16=True):
    """float64 forward (head not applied) and the error scale of the output in units of 2^-24, as
    test_policy_routes_gpu.py ``_net64``; the fp16-split term is included whichever route the pair takes"""
    h, E = x, torch.zeros_like(x)
    for l, (W, b) in enumerate(layers):
        Wa, ha = W.abs(), h.abs()
        z = h @ W.T + b
        E = E @ Wa.T + ha @ Wa.T + b.abs()
        if f16 and l > 0:
            E = E + 2.0 ** -14 * float(Wa.max()) * ha.sum(1, keepdim=True)
        if l + 1 < len(layers):
            h, E = torch.tanh(z), E + TANH_UNITS
    return z, E


def _mean64(agent, actor_flat, x):
    """the actor mean in float64 and its scale (test_policy_routes_gpu.py ``_reference``)"""
    z, Ez = _net64(_layers64(agent.actor, actor_flat), x)
    lo, hi = agent.policy.a_min.double(), agent.policy.a_max.double()
    head = agent.policy.out_act
    if head == 1:
        return torch.relu(z), Ez
    if head == 0:
        return z, Ez
    off = (lo + hi) / 2
    mean = torch.tanh(z) * (hi - off) + off
    return mean, (hi - off) * (Ez + TANH_UNITS + 1) + off.abs() + mean.abs()


def _ratio(err, scale):
    return float((err.abs() / (EPS32 * scale + 1e-300)).max()) if err.numel() else 0.0


def _rel(got, ref):
    return float((got.double() - ref.double()).abs().max() / max(float(ref.double().abs().max()), 1e-300))


def _time_major(x):
    """[T, D, N] -> [T * N, D] in (t, instance) order: sample b = t * N + i"""
    T, D, N = x.shape
    return x.permute(0, 2, 1).reshape(T * N, D)


# ------------------------------------------------------------------------------------------------ the state
def snapshot(agent):
    """everything of the agent a PPO2 iteration reads, taken before collect()"""
    st = {"actor_mod": agent.actor, "critic_mod": agent.critic, "actor": _flat(agent.actor).clone(),
          "critic": _flat(agent.critic).clone(), "key": agent._epoch_key, "total_steps": agent.total_steps,
          "std": agent.std.clone(), "msg": dict(agent.msg), "timeout": agent.buffer.timeout_flag}
    if agent.fused is not None:
        f = agent.fused
        st.update(learner="fused", exp_avg=f.exp_avg.clone(), exp_avg_sq=f.exp_avg_sq.clone(), step=f.step_count,
                  lr=list(f.lr))
    else:
        st.update(learner="torch", gen=agent._gen.get_state(), lr=[agent.optimizer_actor.param_groups[0]["lr"],
                                                                   agent.optimizer_critic.param_groups[0]["lr"]])
        st.update(torch_adam_state(agent))
    if agent.reward_norm is not None:
        st["run"] = agent.reward_norm._run.cpu().numpy().copy()
    return st


def torch_adam_state(agent):
    ms, vs, steps = [], [], set()
    for net, opt in ((agent.actor, agent.optimizer_actor), (agent.critic, agent.optimizer_critic)):
        for lin in _linears(net):
            for p in (lin.weight, lin.bias):
                s = opt.state.get(p, {})
                ms.append(s["exp_avg"].reshape(-1).clone() if s else torch.zeros(p.numel(), device=p.device))
                vs.append(s["exp_avg_sq"].reshape(-1).clone() if s else torch.zeros(p.numel(), device=p.device))
                steps.add(int(s["step"]) if s else 0)
    assert len(steps) == 1, steps
    return {"exp_avg": torch.cat(ms), "exp_avg_sq": torch.cat(vs), "step": steps.pop()}


def capture_raw_rewards(agent):
    """wrap reward_norm.normalize_rows so that it keeps a copy of its input: the raw reward column of every collect()"""
    norm, raw = agent.reward_norm, {}
    orig = norm.normalize_rows

    def normalize_rows(x, out=None):
        raw["r"] = x.clone()
        return orig(x, out=out)
    norm.normalize_rows = normalize_rows
    return raw


def rollout(agent, raw):
    buf = agent.buffer
    r = raw.pop("r") if agent.reward_norm is not None else buf.r.clone()
    return {"s": buf.s.clone(), "s_": buf.s_.clone(), "a": buf.a.clone(), "a_lp": buf.a_lp.clone(), "r_raw": r,
            "r": buf.r.clone(), "done": buf.done.clone(), "flag": buf.flag.clone()}


# ------------------------------------------------------------------------------------------------ the restatement
def reward_rows(run, raws):
    """step 1 in numpy float64: ``run`` = (n, mean, S) [3, 1]; ``raws`` = each rank's [T, N] raw rewards.  Returns each
    rank's normalised rows (float64), the statistics after every row, and the final state."""
    from reinforcementlearningplatform_b200.normalization import merge_stats_reference
    n, mean, S = (np.asarray(v, dtype=np.float64).reshape(-1)[:1] for v in run)
    xs = [np.asarray(r.double().cpu().numpy(), dtype=np.float64) for r in raws]
    outs = [np.empty_like(x) for x in xs]
    rows = []
    for t in range(xs[0].shape[0]):
        batches = []
        for x in xs:
            m = x[t].mean() if x.shape[1] > 1 else x[t, 0]
            batches.append((np.float64(x.shape[1]), m, ((x[t] - m) ** 2).sum() if x.shape[1] > 1 else np.float64(0)))
        n, mean, S = merge_stats_reference((n, mean, S), batches)
        std = mean if float(n[0]) == 1 else np.sqrt(S / n)
        for x, o in zip(xs, outs):
            o[t] = (x[t] - mean) / (std + 1e-8)
        rows.append((float(mean[0]), float(std[0])))
    return outs, rows, (n, mean, S)


def gae_statement(r, vs, vs_, done, flag, timeout, gamma, lmd):
    """PPO2.py:88-98 on [T, N] tensors of one dtype: adv, v_target, and the absolute-value pass of the same scan (the
    scale of its rounding)"""
    succ = ((done != 0) & (flag != timeout)).to(r.dtype)
    dn = (done != 0).to(r.dtype)
    deltas = r + gamma * (1 - succ) * vs_ - vs
    adv = torch.zeros_like(r)
    sc = torch.zeros_like(r, dtype=torch.float64)
    g = torch.zeros_like(r[0])
    s = torch.zeros_like(sc[0])
    for t in range(r.shape[0] - 1, -1, -1):
        g = deltas[t] + gamma * lmd * g * (1 - dn[t])
        adv[t] = g
        s = (r[t].abs() + gamma * (1 - succ[t]) * vs_[t].abs() + vs[t].abs() + deltas[t].abs()).double() \
            + g.abs().double() + gamma * lmd * (1 - dn[t]).double() * s
        sc[t] = s
    return adv, adv + vs, sc


def adv_normalize(advs):
    """(adv - mean) / (std + 1e-5) over all ranks' samples, std unbiased (two-pass)"""
    n = sum(a.numel() for a in advs)
    mean = sum(a.sum() for a in advs) / n
    std = torch.sqrt(sum(((a - mean) ** 2).sum() for a in advs) / (n - 1))
    return [(a - mean) / (std + 1e-5) for a in advs], mean, std


def lr_decay_statement(m, lr, total_steps):
    """PPO2.py:162-171: linear decay to total_steps / max_train_steps, floored at 1e-6; from max_train_steps on the
    learning rates stay where they are"""
    if m["use_lr_decay"] and total_steps < m["max_train_steps"]:
        f = 1 - total_steps / m["max_train_steps"]
        return [max(m["a_lr"] * f, 1e-6), max(m["c_lr"] * f, 1e-6)]
    return list(lr)


def restate_rewards(st, ranks):
    """step 1: each rank's normalised rewards (float64), the statistics after every row and the final state"""
    if "run" not in st:
        return {"r": [d["r_raw"].double() for d in ranks]}
    rn, rows, run = reward_rows(st["run"], [d["r_raw"] for d in ranks])
    return {"r": [torch.as_tensor(x, device=ranks[0]["r_raw"].device) for x in rn], "reward_rows": rows, "run": run}


def restate_iteration(st, ranks, dtype, n_mb=None):
    """One PPO2 iteration from the state ``st`` (``snapshot``) on each rank's rollout ``ranks`` (``rollout``), in
    ``dtype``.  ``n_mb``: the mini-batch count agreed over ranks (two ranks)."""
    m = st["msg"]
    dev = st["actor"].device
    world = len(ranks)
    T, S, N0 = ranks[0]["s"].shape
    gamma, lmd, K, eps_clip = m["gamma"], m["lmd"], m["K_epochs"], m["eps_clip"]
    actor, critic = copy.deepcopy(st["actor_mod"]).to(dtype), copy.deepcopy(st["critic_mod"]).to(dtype)
    _load_flat(actor, st["actor"].to(dtype))
    _load_flat(critic, st["critic"].to(dtype))
    std = st["std"].to(dtype)
    # 1. rewards
    res = restate_rewards(st, ranks)
    rs = res["r"]
    # 2. values and advantages
    advs, vts, flat = [], [], []
    with torch.no_grad():
        for d, r in zip(ranks, rs):
            T, S, N = d["s"].shape
            vs = critic(_time_major(d["s"]).to(dtype)).reshape(T, N)
            vs_ = critic(_time_major(d["s_"]).to(dtype)).reshape(T, N)
            adv, vt, _ = gae_statement(r.to(dtype), vs, vs_, d["done"], d["flag"], st["timeout"], gamma, lmd)
            advs.append(adv)
            vts.append(vt)
    if m["use_adv_norm"]:
        advs, res["adv_mean"], res["adv_std"] = adv_normalize(advs)
    res["adv"], res["v_target"] = advs, vts
    for d, adv, vt in zip(ranks, advs, vts):
        flat.append({"s": _time_major(d["s"]).to(dtype), "a": _time_major(d["a"]).to(dtype),
                     "a_lp": _time_major(d["a_lp"]).to(dtype).sum(1, keepdim=True),
                     "adv": adv.reshape(-1, 1), "v_target": vt.reshape(-1, 1)})
    # 3. index sets
    Bs = [f["s"].shape[0] for f in flat]
    mb = [min(m["mini_batch_size"], B) if m["using_mini_batch"] else B for B in Bs]
    if n_mb is None:
        n_mb = min(-(-B // b) for B, b in zip(Bs, mb))
    if st["learner"] == "fused":
        sets = [fused_index_sets(st["key"], B, b, n_mb, K, world > 1) for B, b in zip(Bs, mb)]
        res["key"] = (st["key"] + K) & (2 ** 64 - 1)
    else:
        assert world == 1
        s0, res["gen"] = torch_index_sets(st["gen"], dev, Bs[0], mb[0], n_mb, K)
        sets = [s0]
    # 4. the update: torch.optim.Adam re-synced to the agent's moments and step
    eps = 1e-5 if m["set_adam_eps"] else 1e-8
    opts = []
    o = 0
    for net, lr in ((actor, st["lr"][0]), (critic, st["lr"][1])):
        params = [t for lin in _linears(net) for t in (lin.weight, lin.bias)]
        opt = torch.optim.Adam(params, lr=lr, eps=eps, foreach=False)
        for p in params:
            k = p.numel()
            opt.state[p] = {"step": torch.tensor(float(st["step"])),
                            "exp_avg": st["exp_avg"][o:o + k].to(dtype).view_as(p).clone(),
                            "exp_avg_sq": st["exp_avg_sq"][o:o + k].to(dtype).view_as(p).clone()}
            o += k
        opts.append(opt)
    head_z = {}
    relu = getattr(st["actor_mod"], "out_act", None) == "relu"
    hook = _linears(actor)[-1].register_forward_hook(lambda mod, i, out: head_z.__setitem__("z", out.detach()))
    n_kink, norms = 0, [[], []]
    for e in range(K):
        for j in range(n_mb):
            actor_loss = 0
            for f, sets_r in zip(flat, sets):
                idx = torch.as_tensor(sets_r[e][j], device=dev)
                mean = actor(f["s"][idx])
                dist_now = torch.distributions.Normal(mean, std.expand_as(mean))
                ent = dist_now.entropy().sum(1, keepdim=True)
                lp_now = dist_now.log_prob(f["a"][idx])
                ratios = torch.exp(lp_now.sum(1, keepdim=True) - f["a_lp"][idx])
                surr1 = ratios * f["adv"][idx]
                surr2 = torch.clamp(ratios, 1 - eps_clip, 1 + eps_clip) * f["adv"][idx]
                loss_r = (-torch.min(surr1, surr2) - m["entropy_coef"] * ent).mean()
                actor_loss = actor_loss + loss_r / world
                r_ = ratios.detach().reshape(-1)
                kink = ((r_ - (1 - eps_clip)).abs() <= KINK) | ((r_ - (1 + eps_clip)).abs() <= KINK)
                if relu:
                    kink |= (head_z["z"].abs() <= KINK).any(1)
                n_kink += int(kink.sum())
            opts[0].zero_grad()
            actor_loss.backward()
            if m["use_grad_clip"]:
                norms[0].append(float(torch.nn.utils.clip_grad_norm_(actor.parameters(), 0.5)))
            opts[0].step()
            critic_loss = 0
            for f, sets_r in zip(flat, sets):
                idx = torch.as_tensor(sets_r[e][j], device=dev)
                critic_loss = critic_loss + torch.nn.functional.mse_loss(f["v_target"][idx], critic(f["s"][idx])) / world
            opts[1].zero_grad()
            critic_loss.backward()
            if m["use_grad_clip"]:
                norms[1].append(float(torch.nn.utils.clip_grad_norm_(critic.parameters(), 0.5)))
            opts[1].step()
            res["loss"] = [float(actor_loss.detach()), float(critic_loss.detach())]
    hook.remove()
    # 5. learning-rate decay: total_steps counts the env steps of the whole group
    res["lr"] = lr_decay_statement(m, st["lr"], st["total_steps"] + sum(Bs))
    res.update(actor=_flat(actor), critic=_flat(critic), n_kink=n_kink, n_mb=n_mb, step=st["step"] + K * n_mb,
               grad_norms=norms)
    states = [opts[k].state[p] for k, net in enumerate((actor, critic)) for lin in _linears(net)
              for p in (lin.weight, lin.bias)]
    res["exp_avg"] = torch.cat([s["exp_avg"].reshape(-1) for s in states])
    res["exp_avg_sq"] = torch.cat([s["exp_avg_sq"].reshape(-1) for s in states])
    return res


# ------------------------------------------------------------------------------------------------ stage checks
def check_collect(agent, st, d, ref, rank=0):
    """actions inside the clamp, log-probs of the pre-iteration actor, normalised rewards of step 1"""
    out = {}
    lo = agent.policy.a_min.view(1, -1, 1)
    hi = agent.policy.a_max.view(1, -1, 1)
    assert bool(((d["a"] >= lo) & (d["a"] <= hi)).all()), "collect(): an action outside the clamp"
    x = _time_major(d["s"]).double()
    mean, Em = _mean64(agent, st["actor"], x)
    a = _time_major(d["a"]).double()
    sd = st["std"].double().expand(a.shape[1])
    dd = a - mean
    lp = -dd * dd / (2 * sd * sd) - torch.log(sd) - 0.5 * math.log(2 * math.pi)
    El = dd.abs() / (sd * sd) * (2 * Em + a.abs() + dd.abs()) + 4 * (dd * dd / (2 * sd * sd) + torch.log(sd).abs() + 1.0)
    out["a_lp"] = _ratio(_time_major(d["a_lp"]).double() - lp, El)
    if "run" in st:
        r64 = ref["r"][rank]
        mean_t = torch.tensor([m for m, _ in ref["reward_rows"]], dtype=torch.float64, device=r64.device).view(-1, 1)
        std_t = torch.tensor([s for _, s in ref["reward_rows"]], dtype=torch.float64, device=r64.device).view(-1, 1)
        scale = r64.abs() + 2.0 ** -29 * (d["r_raw"].double().abs() + mean_t.abs()) / (std_t + 1e-8).abs()
        out["r"] = _ratio(d["r"].double() - r64, scale)
    return out


def check_values_and_gae(agent, st, d):
    """V(s), V(s') of learn()'s critic-only K-POLICY launches against the float64 critic; buf.gae on those values against
    the GAE statement in float64 on the same values"""
    buf, m = agent.buffer, agent.msg
    T, S, N = d["s"].shape
    vs = torch.empty(T, N, device=d["s"].device)
    vs_ = torch.empty_like(vs)
    for t in range(T):
        agent.value_net(buf.s[t], value=vs[t])
        agent.value_net(buf.s_[t], value=vs_[t])
    layers = _layers64(agent.critic, st["critic"])
    out = {}
    for name, got, src in (("V(s)", vs, d["s"]), ("V(s')", vs_, d["s_"])):
        z, E = _net64(layers, _time_major(src).double())
        out[name] = _ratio(got.reshape(-1).double() - z[:, 0], E[:, 0])
    adv, vt = buf.gae(vs, vs_, agent.gamma, agent.lmd, normalize=m["use_adv_norm"])
    a64, vt64, sc = gae_statement(d["r"].double(), vs.double(), vs_.double(), d["done"], d["flag"], st["timeout"],
                                  agent.gamma, agent.lmd)
    out["v_target"] = _ratio(vt.double() - vt64, sc + vs.double().abs() + vt64.abs())
    if m["use_adv_norm"]:
        (an,), mean, sd = adv_normalize([a64])
        den = sd + 1e-5
        scale = (sc + mean.abs() + sc.mean()) / den + an.abs()
        out["adv"] = _ratio(adv.double() - an, scale)
        out["|mean|/std"] = float(mean.abs() / sd)
    else:
        out["adv"] = _ratio(adv.double() - a64, sc)
    return out


def check_learn(agent, st, res, res32, out_loss):
    """parameters, Adam moments, step, returned losses, learning rates, key / generator after learn()"""
    out, f32 = {}, {}
    nets = (("actor", agent.actor), ("critic", agent.critic))
    for k, (name, net) in enumerate(nets):
        out[f"{name} param"] = float((_flat(net).double() - res[name]).abs().max())
        f32[f"{name} param"] = float((res32[name].double() - res[name]).abs().max())
    if agent.fused is not None:
        ea, eas, step, lr = agent.fused.exp_avg, agent.fused.exp_avg_sq, agent.fused.step_count, list(agent.fused.lr)
    else:
        s = torch_adam_state(agent)
        ea, eas, step = s["exp_avg"], s["exp_avg_sq"], s["step"]
        lr = [agent.optimizer_actor.param_groups[0]["lr"], agent.optimizer_critic.param_groups[0]["lr"]]
    na = st["actor"].numel()
    for name, got, ref, r32 in (("exp_avg", ea, res["exp_avg"], res32["exp_avg"]),
                                ("exp_avg_sq", eas, res["exp_avg_sq"], res32["exp_avg_sq"])):
        for part, sl in (("actor", slice(0, na)), ("critic", slice(na, None))):
            out[f"{part} {name}"] = _rel(got[sl], ref[sl])
            f32[f"{part} {name}"] = _rel(r32[sl], ref[sl])
    assert step == res["step"], (step, res["step"])
    assert lr == res["lr"], (lr, res["lr"])
    if agent.fused is not None:
        assert agent._epoch_key == res["key"], "the permutation key did not advance by K_epochs"
    else:
        assert torch.equal(agent._gen.get_state(), res["gen"]), "the generator is not where K_epochs randperms leave it"
    if out_loss is not None:
        for k, name in enumerate(("actor_loss", "critic_loss")):
            den = max(abs(res["loss"][k]), 1e-30)
            out[name] = abs(out_loss[name] - res["loss"][k]) / den
            f32[name] = abs(res32["loss"][k] - res["loss"][k]) / den
    return out, f32


def check_packed(agent, obs):
    """evaluate() on the next rollout's first row follows the updated actor (K-POLICY's packed copy was refreshed)"""
    got = agent.evaluate(obs).double().T
    mean, Em = _mean64(agent, _flat(agent.actor), obs.double().T)
    act = torch.minimum(torch.maximum(mean, agent.policy.a_min.double()), agent.policy.a_max.double())
    return _ratio(got - act, Em + act.abs())


def _assert_bounds(tag, r):
    for k, v in r.items():
        if k != "|mean|/std":
            b = _bound(k)
            assert v <= b, (tag, k, v, b)


def _bound(k):
    bounds = {"a_lp": C_LP, "r": C_REWARD, "V(s)": C_VALUE, "V(s')": C_VALUE, "v_target": C_GAE, "adv": C_GAE,
              "evaluate": C_LP, "actor param": PARAM_TOL[0], "critic param": PARAM_TOL[1], "actor exp_avg": MOMENT_TOL,
              "critic exp_avg": MOMENT_TOL, "actor exp_avg_sq": MOMENT_TOL, "critic exp_avg_sq": MOMENT_TOL,
              "actor_loss": LOSS_TOL, "critic_loss": LOSS_TOL}
    return bounds[k.split(" rank")[0]]


# ------------------------------------------------------------------------------------------------ the cases
def _cartpole(n, seed=3, learner="auto", msg=None, reward_norm=True, std=0.8):
    import reinforcementlearningplatform_b200 as rlp
    from reinforcementlearningplatform_b200.ppo2 import VecPPO2, reference_nets
    env = rlp.CartPoleAngleOnly(n_envs=n, variant="ppo2", io_dtype=torch.float32, auto_reset=True, seed=seed)
    torch.manual_seed(11)
    actor, critic = reference_nets(env.state_dim, env.action_dim, "cuda", init_std=std, mean_act="identity")
    return VecPPO2(env, actor, critic, msg, std=std, seed=seed, learner=learner, reward_norm=reward_norm)


def _uav(n):
    import reinforcementlearningplatform_b200 as rlp
    from reinforcementlearningplatform_b200.ppo2 import VecPPO2, reference_nets
    env = rlp.UavPosCtrlRL(n_envs=n, random_trajectory=True, io_dtype=torch.float32, auto_reset=True, seed=4)
    torch.manual_seed(12)
    actor, critic = reference_nets(env.state_dim, env.action_dim, "cuda", init_std=0.45)
    with torch.no_grad():   # relu head: every pre-activation well away from the kink, half the units inactive
        actor.mean_layer.bias.copy_(torch.tensor([0.5, -0.5] * (env.action_dim // 2), device="cuda"))
    msg = {"buffer_size": 16, "K_epochs": 3, "using_mini_batch": False, "max_train_steps": int(1e7)}
    return VecPPO2(env, actor, critic, msg, std=0.45, reward_norm=False, seed=1)


def _soi(n):
    import reinforcementlearningplatform_b200 as rlp
    from reinforcementlearningplatform_b200.ppo2 import VecPPO2, dppo2_nets
    env = rlp.SecondOrderIntegration(n_envs=n, variant="dppo2", io_dtype=torch.float32, auto_reset=True, seed=5)
    torch.manual_seed(13)
    ar = np.asarray(env.action_range, dtype=np.float32)
    actor, critic = dppo2_nets(env.state_dim, env.action_dim, ar[:, 0], ar[:, 1], "cuda", hidden=64)
    msg = {"buffer_size": 16, "K_epochs": 3, "mini_batch_size": 3000, "entropy_coef": 0.0, "use_grad_clip": False,
           "use_adv_norm": False, "use_lr_decay": False}
    return VecPPO2(env, actor, critic, msg, seed=2)


def _ugvo(n):
    import reinforcementlearningplatform_b200 as rlp
    from reinforcementlearningplatform_b200.ppo2 import VecPPO2, dppo2_nets
    env = rlp.UGVForwardObstacleAvoidance(n_envs=n, variant="dppo2", io_dtype=torch.float32, auto_reset=True, seed=6)
    torch.manual_seed(14)
    ar = np.asarray(env.action_range, dtype=np.float32)
    actor, critic = dppo2_nets(env.state_dim, env.action_dim, ar[:, 0], ar[:, 1], "cuda", hidden=256)
    msg = {"buffer_size": 16, "K_epochs": 3, "mini_batch_size": 100000, "max_train_steps": int(1e6)}
    return VecPPO2(env, actor, critic, msg, seed=3)


CASE_A_MSG = {"buffer_size": 7, "K_epochs": 3, "mini_batch_size": 2333, "max_train_steps": 14001}
CASES = {
    # name: (agent factory, iterations, between-iterations hook)
    "a_cartpole_last_batch_of_one": (lambda: _cartpole(1000, msg=CASE_A_MSG), 3, None),
    "b_uav_raw_rewards_one_batch": (lambda: _uav(2048), 2, None),
    "c_soi_tanh_range_std_vector": (lambda: _soi(512), 2, lambda ag, it: ag.set_action_std(ag.std.cpu().numpy() * 0.7)),
    "d_cartpole_single_instance": (lambda: _cartpole(1, msg={"buffer_size": 64, "K_epochs": 3}), 3, None),
    "e_cartpole_torch_learner": (lambda: _cartpole(1000, learner="torch", msg=CASE_A_MSG), 3, None),
    "f_ugvo_dppo2_256_torch": (lambda: _ugvo(512), 2, None),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_ppo2_iterations_match_the_float64_restatement(case):
    make, iters, between = CASES[case]
    agent = make()
    assert (agent.fused is None) == (case[0] in "ef"), "the case must reach its learner"
    raw = capture_raw_rewards(agent) if agent.reward_norm is not None else {}
    agent.env.reset(True)
    lines, worst = [], {}
    for it in range(iters):
        if between is not None and it > 0:
            between(agent, it)
        st = snapshot(agent)
        agent.collect()
        d = rollout(agent, raw)
        res = restate_iteration(st, [d], torch.float64)
        res32 = restate_iteration(st, [d], torch.float32)
        r = check_collect(agent, st, d, res)
        if case.startswith("d"):
            check_single_instance_rewards(agent, st, d, res)
        r.update(check_values_and_gae(agent, st, d))
        out = agent.learn()
        lr_used = list(st["lr"])
        rl, f32 = check_learn(agent, st, res, res32, out)
        r.update(rl)
        r["evaluate"] = check_packed(agent, agent.env._reset_obs)
        assert res["n_kink"] == 0, ("samples at a clip edge or relu kink", res["n_kink"])
        lines.append(f"  it {it}: lr {lr_used} -> {res['lr']}, mini-batches {res['n_mb']} x {st['msg']['K_epochs']}, "
                     + "  ".join(f"{k} {v:.3g}" for k, v in r.items())
                     + "  | float32 restatement: " + "  ".join(f"{k} {v:.3g}" for k, v in f32.items()))
        print(f"\n{case}" + lines[-1], flush=True)
        for k, v in r.items():
            worst[k] = max(worst.get(k, 0.0), v)
        _assert_bounds(f"{case} it {it}", r)
    # the agent's next rollout samples with the updated actor: its log-probs follow it (check_collect of one more)
    st = snapshot(agent)
    agent.collect()
    d = rollout(agent, raw)
    worst["next a_lp"] = check_collect(agent, st, d, restate_rewards(st, [d]))["a_lp"]
    print(f"\n{case}:\n" + "\n".join(lines) + "\n  worst: " + "  ".join(f"{k} {v:.3g}" for k, v in worst.items()))
    assert worst["next a_lp"] <= C_LP, worst["next a_lp"]
    if case.startswith("a") or case.startswith("e"):
        # lr factors 1 -> ~1/2 -> the 1e-6 floor (total_steps 14000 of 14001) -> past max_train_steps: unchanged
        m = agent.msg
        assert agent.total_steps == 4 * 7000
        lr = agent.fused.lr if agent.fused is not None else [agent.optimizer_actor.param_groups[0]["lr"],
                                                             agent.optimizer_critic.param_groups[0]["lr"]]
        assert lr == [1e-6, 1e-6], lr
        assert m["max_train_steps"] == 14001


def check_single_instance_rewards(agent, st, d, res):
    """N = 1: every reward row is a batch of one, so the running statistics are the reference's sample-by-sample
    recurrence (b200_norm_seq, pinned to tests/golden/norm.npz by test_norm.py) bit for bit, and so are the rewards"""
    from reinforcementlearningplatform_b200.normalization import Normalization
    seq = Normalization(1, device="cuda")
    seq._run.copy_(torch.as_tensor(st["run"], device="cuda"))
    y = seq.seq(d["r_raw"].reshape(1, -1).contiguous())
    assert torch.equal(y.reshape(-1), d["r"].reshape(-1)), "normalised rewards differ from the reference recurrence"
    assert torch.equal(seq._run, agent.reward_norm._run), "running statistics differ from the reference recurrence"
    n, mean, S = res["run"]
    run = agent.reward_norm._run.cpu().numpy().reshape(-1)
    assert (run[0], run[1], run[2]) == (n[0], mean[0], S[0]), (run, n, mean, S)
    assert torch.equal(res["r"][0].float(), d["r"]), "the float64 statement rounded to float32 differs"


# ------------------------------------------------------------------------------------------------ CPU: the index sets
def test_restated_index_sets_cover_every_sample_once_per_epoch():
    """the restatement's mini-batches: case a's 7000 = 3 x 2333 + 1 (last batch of one sample), the two-rank even split
    of 16,400 samples into the agreed 4 batches, and a new permutation every epoch"""
    sets = fused_index_sets(12345, 7000, 2333, 4, 3)
    assert [len(x) for x in sets[0]] == [2333, 2333, 2333, 1]
    for e in sets:
        assert np.array_equal(np.sort(np.concatenate(e)), np.arange(7000))
    assert not np.array_equal(sets[0][0], sets[1][0])
    assert np.array_equal(sets[1][0], keyed_positions(12346, 7000, 0, 2333))
    assert mini_batch_bounds(16400, 4096, 4, grouped=True) == [0, 4100, 8200, 12300, 16400]
    assert mini_batch_bounds(16384, 4096, 4, grouped=True) == [0, 4096, 8192, 12288, 16384]
    assert mini_batch_bounds(7000, 2333, 4) == [0, 2333, 4666, 6999, 7000]
    # a rank whose own count equals the agreed one still splits evenly (the two-rank test's second iteration)
    assert mini_batch_bounds(16384, 4099, 4, grouped=True) == [0, 4096, 8192, 12288, 16384]
    assert mini_batch_bounds(16384, 4099, 4) == [0, 4099, 8198, 12297, 16384]
    split = fused_index_sets(7, 16400, 4096, 4, 2, grouped=True)
    for e in split:
        assert [len(x) for x in e] == [4100] * 4
        assert np.array_equal(np.sort(np.concatenate(e)), np.arange(16400))


def test_reward_rows_restatement_is_the_reference_recurrence_for_one_instance():
    """reward_rows with N = 1 is RunningMeanStd fed one sample at a time (utils/classes.py:626-656), n == 1 quirk
    included, in float64"""
    x = np.array([[0.5], [-1.25], [3.0], [0.0], [7.5]], dtype=np.float32)
    (out,), _, (n, mean, S) = reward_rows(np.zeros((3, 1)), [torch.as_tensor(x)])
    rn, rm, rs, ys = 0, 0.0, 0.0, []
    for v in x[:, 0].astype(np.float64):
        rn += 1
        if rn == 1:
            rm, std = v, v
        else:
            old = rm
            rm = old + (v - old) / rn
            rs = rs + (v - old) * (v - rm)
            std = np.sqrt(rs / rn)
        ys.append((v - rm) / (std + 1e-8))
    assert (float(n[0]), float(mean[0]), float(S[0])) == (rn, rm, rs)
    assert np.array_equal(out[:, 0], np.array(ys))


# ------------------------------------------------------------------------------------------------ two ranks
N_SHARDS = 2049          # shards of 1025 and 1024 instances
TWO_RANK_MSG = {"buffer_size": 16, "K_epochs": 2, "mini_batch_size": 4096}


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _cpu(x):
    if torch.is_tensor(x):
        return x.detach().cpu()
    if isinstance(x, dict):
        return {k: _cpu(v) for k, v in x.items() if k not in ("actor_mod", "critic_mod")}
    return x


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK="0")
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    torch.cuda.set_device(0)
    dist.init_process_group("gloo")
    import reinforcementlearningplatform_b200 as rlp
    from reinforcementlearningplatform_b200 import dist as D
    from reinforcementlearningplatform_b200.ppo2 import VecPPO2, reference_nets
    n_local, off = D.shard(N_SHARDS, rank, world)
    env = rlp.CartPoleAngleOnly(n_envs=n_local, variant="ppo2", io_dtype=torch.float32, auto_reset=True, seed=3,
                                env_index_offset=off)
    torch.manual_seed(100 + rank)                        # different initial weights: rank 0's are broadcast
    actor, critic = reference_nets(env.state_dim, env.action_dim, "cuda", init_std=0.8, mean_act="identity")
    agent = VecPPO2(env, actor, critic, TWO_RANK_MSG, std=0.8, seed=7, group=None)
    raw = capture_raw_rewards(agent)
    env.reset(True)
    its = []
    for it in range(2):
        if it == 1:   # rank 1's B = 16384 is no multiple of 4099 and its own ceil(B / mb) = 4 is the agreed count
            agent.msg["mini_batch_size"] = 4099
        st = snapshot(agent)
        agent.collect()
        d = rollout(agent, raw)
        agent.learn()
        after = snapshot(agent)
        its.append((_cpu(st), _cpu(d), _cpu(after), agent._epoch_key))
    q.put(pickle.dumps((rank, n_local, its)))      # by value: the worker exits before the parent reads
    dist.destroy_process_group()


@pytest.mark.gpu
def test_two_ranks_match_the_data_parallel_restatement():
    import torch.multiprocessing as mp
    import reinforcementlearningplatform_b200 as rlp
    from reinforcementlearningplatform_b200.ppo2 import reference_nets
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted((pickle.loads(q.get(timeout=600)) for _ in procs), key=lambda x: x[0])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    (_, n0, its0), (_, n1, its1) = res
    assert (n0, n1) == (1025, 1024)
    env = rlp.CartPoleAngleOnly(n_envs=1, variant="ppo2", io_dtype=torch.float32)
    actor, critic = reference_nets(env.state_dim, env.action_dim, "cuda", mean_act="identity")
    lines = []
    for it in range(2):
        (st0, d0, a0, key0), (st1, d1, a1, key1) = its0[it], its1[it]
        for k in ("actor", "critic", "exp_avg", "exp_avg_sq", "run"):       # the ranks start from one state
            assert np.array_equal(np.asarray(st0[k]), np.asarray(st1[k])), k
        assert st0["lr"] == st1["lr"] and st0["total_steps"] == st1["total_steps"] == N_SHARDS * 16 * it
        st = {k: (v.cuda() if torch.is_tensor(v) else v) for k, v in st0.items()}
        st.update(actor_mod=actor, critic_mod=critic)
        ranks = [{k: v.cuda() for k, v in d.items()} for d in (d0, d1)]
        # rank 0 alone would run ceil(16400 / mb) = 5 mini-batches, rank 1 4: the agreed count is 4 (mb 4096, then 4099)
        ref = restate_iteration(st, ranks, torch.float64)
        ref32 = restate_iteration(st, ranks, torch.float32)
        assert ref["n_mb"] == 4 and ref["n_kink"] == 0
        r = {}
        for rank, d in enumerate(ranks):
            T = d["r"].shape[0]
            mean_t = torch.tensor([m for m, _ in ref["reward_rows"]], dtype=torch.float64, device="cuda").view(T, 1)
            std_t = torch.tensor([s for _, s in ref["reward_rows"]], dtype=torch.float64, device="cuda").view(T, 1)
            r64 = ref["r"][rank]
            scale = r64.abs() + 2.0 ** -29 * (d["r_raw"].double().abs() + mean_t.abs()) / (std_t + 1e-8).abs()
            r[f"r rank {rank}"] = _ratio(d["r"].double() - r64, scale)
        f32 = {}
        na = st["actor"].numel()
        for rank, a in enumerate((a0, a1)):
            # one learning rate on every rank, decayed with the group's step count
            assert a["step"] == ref["step"] and a["lr"] == ref["lr"], (rank, a["lr"], ref["lr"])
            assert a["total_steps"] == N_SHARDS * 16 * (it + 1)
            assert (key0, key1)[rank] == ref["key"]
            for name in ("actor", "critic"):
                r[f"{name} param rank {rank}"] = float((a[name].cuda().double() - ref[name]).abs().max())
            for name in ("exp_avg", "exp_avg_sq"):
                for part, sl in (("actor", slice(0, na)), ("critic", slice(na, None))):
                    r[f"{part} {name} rank {rank}"] = _rel(a[name].cuda()[sl], ref[name][sl])
        for name in ("actor", "critic"):
            f32[f"{name} param"] = float((ref32[name].double() - ref[name]).abs().max())
        assert np.array_equal(a0["run"], a1["run"]) and a0["run"][0, 0] == ref["run"][0][0] == N_SHARDS * T * (it + 1)
        lines.append(f"  it {it}: " + "  ".join(f"{k} {v:.3g}" for k, v in r.items())
                     + f"  grad norms actor {max(ref['grad_norms'][0]):.3g} critic {max(ref['grad_norms'][1]):.3g}"
                     + "  | float32 restatement: " + "  ".join(f"{k} {v:.3g}" for k, v in f32.items()))
        print("\ntwo ranks" + lines[-1], flush=True)
        _assert_bounds(f"two ranks it {it}", r)
    print("\ntwo ranks:\n" + "\n".join(lines))
