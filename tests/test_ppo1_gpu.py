"""GPU: the PPO v1 update (b200_mc_returns_stats, b200_ppo1_grad, VecPPO).

The v1 loss is restated here (DESIGN 4), not pinned by a recording of the reference learner:
    R_hat = (R - mean(R)) / (std(R) + 1e-7);  V = critic(s);  adv = R_hat - V (no gradient);
    loss = mean(-min(ratio adv, clamp(ratio, 1 +- eps_clip) adv)) + value_coef mse(V, R_hat) - entropy_coef H.
Checked here: the return statistics against float64 numpy sums; the advantage launch against the critic forward of
K-LEARN's gradient kernel (bit for bit); b200_ppo1_grad against b200_ppo2_grad (bit for bit) and against float64 autograd
of the joint loss within K-LEARN's bound ``C_GRAD * 2^-24 * scale`` (DESIGN 4(d), the helpers restated from
test_learn_gpu.py); VecPPO.learn() against a float32 torch restatement of the loop; training; set_action_std; two ranks."""
import copy
import ctypes as C
import math
import os
import socket
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

EPS32 = 2.0 ** -24
ULP_SUM = 2.0 ** -53
C_GRAD = 48.0        # K-LEARN's bound (DESIGN 4(d)): 10x the largest ratio measured over the PPO2 sweep
C_NORM = 64.0        # R_hat against torch float32, in units of 2^-24 ((|R| + |mean|) / (std + eps) + |R_hat|)
PARAM_TOL = 1e-6     # VecPPO.learn() against the torch restatement, after every epoch (the PPO2 comparison's bound)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _lib():
    from reinforcementlearningplatform_b200 import _lib
    return _lib


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


# ------------------------------------------------------------------------------------------------ 1. return statistics
def _rewards(T, N, dtype, seed, scale=1.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    r = ((torch.rand(T, N, device="cuda", generator=g, dtype=torch.float64) * 2 - 0.7) * scale).to(dtype).contiguous()
    done = (torch.rand(T, N, device="cuda", generator=g) < 0.05).to(torch.uint8).contiguous()
    return r, done


def _ret_stats(r, done, gamma=0.99):
    from reinforcementlearningplatform_b200 import gae
    stats = torch.zeros(3, dtype=torch.float64, device="cuda")
    ret = gae.mc_returns(r, done, gamma, stats=stats)
    return ret, stats


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("N", [1, 127, 128, 129, 100003])
@pytest.mark.parametrize("T", [1, 7, 64, 1000])
def test_return_statistics(T, N, dtype):
    from reinforcementlearningplatform_b200 import gae
    r, done = _rewards(T, N, dtype, seed=T * 7 + N)
    ret, stats = _ret_stats(r, done)
    assert torch.equal(ret, gae.mc_returns(r, done, 0.99))                      # bit-identical to b200_mc_returns
    x = ret.double().cpu().numpy().ravel()
    st = stats.cpu().numpy()
    n = x.size
    assert st[2] == n
    for k, v in ((0, x), (1, x * x)):
        exact = float(v.astype(np.longdouble).sum())
        assert abs(st[k] - exact) <= n * ULP_SUM * float(np.abs(v).astype(np.longdouble).sum()), (k, st[k], exact)
    # the statistics increment: a second call adds the same sums again; a repeated run gives the same bits
    ret2, stats2 = _ret_stats(r, done)
    assert torch.equal(ret2, ret) and torch.equal(stats2, stats)
    gae.mc_returns(r, done, 0.99, stats=stats2)
    assert float(stats2[2]) == 2 * n
    if n > 1 and n <= (1 << 23):
        # R_hat against torch float32 (R - R.mean()) / (R.std() + 1e-7)
        hat = gae.normalize_advantage(ret.clone(), stats.clone(), eps=1e-7)
        den = ret.std() + 1e-7
        ref = (ret - ret.mean()) / den
        scale = (ret.abs() + ret.mean().abs()) / den + ref.abs()
        worst = float(((hat - ref).abs().double() / (EPS32 * scale.double() + 1e-300)).max())
        print(f"\nT={T} N={N} {dtype}: R_hat within {worst:.2f} x 2^-24 of torch float32")
        assert worst <= C_NORM, worst


def test_normalisation_eps_matters_for_small_returns():
    """returns of std ~1e-6: the 1e-7 of (R - mean) / (std + 1e-7) moves R_hat by ~10 %; the kernel keeps it"""
    from reinforcementlearningplatform_b200 import gae
    r, done = _rewards(64, 4099, torch.float32, seed=5, scale=1e-7)
    ret, stats = _ret_stats(r, done)
    hat = gae.normalize_advantage(ret.clone(), stats, eps=1e-7)
    ref = ((ret.double() - ret.double().mean()) / (ret.double().std() + 1e-7)).float()
    no_eps = ((ret.double() - ret.double().mean()) / ret.double().std()).float()
    assert float((hat - ref).abs().max()) <= 1e-5 * float(ref.abs().max())
    assert float((no_eps - ref).abs().max()) >= 0.02 * float(ref.abs().max())


# ------------------------------------------------------------------------------------------------ helpers (K-LEARN's bound)
class _Net(torch.nn.Sequential):
    """nn.Linear layers, tanh between them, ``head`` on the last (identity / relu / tanh_range); keeps every layer's input
    H_l and pre-activation Z_l (the output's gradient retained) for the error bound (test_learn_gpu.py)."""

    def __init__(self, dims, head="identity", gain=None, off=None):
        super().__init__(*[torch.nn.Linear(i, o) for i, o in zip(dims[:-1], dims[1:])])
        self.head, self.gain, self.off = head, gain, off

    def forward(self, x):
        self.H, self.Z = [], []
        for l, lin in enumerate(self):
            self.H.append(x.detach())
            x = lin(x)
            self.Z.append(x)
            if l + 1 < len(self):
                x = torch.tanh(x)
            elif x.requires_grad:
                x.retain_grad()
        if self.head == "relu":
            return torch.relu(x)
        if self.head == "tanh_range":
            as_t = lambda v: torch.as_tensor(v, dtype=x.dtype, device=x.device)
            return torch.tanh(x) * as_t(self.gain) + as_t(self.off)
        return x


def _fwd_scales(net):
    """Hc_l >= |H_l|: the forward pass in absolute value, Hc_0 = |x|, Hc_{l+1} = |H_{l+1}| + (1 - H_{l+1}^2) zc_l with
    zc_l = Hc_l |W_l|^T + |b_l|; also returns zc of the output layer (the condition number of the net's output)"""
    Hc = [net.H[0].abs()]
    zc = None
    for l in range(len(net)):
        zc = Hc[l] @ net[l].weight.detach().abs().t() + net[l].bias.detach().abs()
        if l + 1 < len(net):
            Hc.append(net.H[l + 1].abs() + (1 - net.H[l + 1] ** 2) * zc)
    return Hc, zc


def _grad_scales(net, g_out):
    """per flat gradient entry: G_l^T Hc_l (weights) and sum_s G_l[s] (bias), G_L = g_out, G_{l-1} = (G_l |W_l|)(1 - H_l^2)"""
    Hc, _ = _fwd_scales(net)
    G = g_out
    out = []
    for l in range(len(net) - 1, -1, -1):
        out = [(G.t() @ Hc[l]).reshape(-1), G.sum(0)] + out
        if l > 0:
            G = (G @ net[l].weight.detach().abs()) * (1 - net.H[l] ** 2)
    return torch.cat(out)


def _out_scale(actor, t):
    """G_L of the actor: dZ_L = c (act - m) / var * dm/dz in absolute value, plus the log-prob rounding inside the ratio"""
    z = actor.Z[-1].detach()
    if actor.head == "relu":
        dmdz = dmdz_abs = (z > 0).to(z.dtype)
    elif actor.head == "tanh_range":
        gain, th = torch.as_tensor(actor.gain, dtype=z.dtype, device=z.device), torch.tanh(z)
        dmdz, dmdz_abs = gain * (1 - th * th), gain * (1 + th * th)
    else:
        dmdz = dmdz_abs = torch.ones_like(z)
    diff = t["act"] - t["mean"]
    g = t["c"].abs() / t["var"] * (diff.abs() * dmdz_abs + (t["act"].abs() + t["mean"].abs()) * dmdz)
    return g + actor.Z[-1].grad.abs() * t["lp_abs"]


def _ratio(err, scale):
    return float((err.abs() / (EPS32 * scale + 1e-30)).max())


def _flat_grads(net):
    return torch.cat([p.grad.reshape(-1) for lin in net for p in (lin.weight, lin.bias)])


# ------------------------------------------------------------------------------------------------ the cases of items 2-4
# actor dims, critic dims, actor head, per-dimension std vector
PAIRS = {
    "ref_relu": ((6, 64, 64, 32, 8), (6, 64, 32, 1), "relu", False),
    "dppo2_64": ((41, 64, 64, 2), (41, 64, 64, 1), "tanh_range", True),
    "w8": ((3, 8, 8, 2), (3, 8, 1), "relu", False),
    "one_layer": ((5, 3), (5, 1), "identity", False),
}
# name -> (how the samples are picked, T, N, first, count), as in test_learn_gpu.py
BATCHES = {
    "i1": ("index", 4, 1000, 17, 1),
    "i63": ("index", 4, 1000, 17, 63),
    "r65": ("repeat", 4, 1000, 17, 65),
    "i3001": ("index", 4, 1000, 17, 3001),
    "p64k": ("perm", 32, 1 << 14, 0, 1 << 16),
    "p512k": ("perm", 32, 1 << 14, 0, 1 << 19),
}
CASES = [(p, b) for p in PAIRS for b in BATCHES]
VALUE_COEFS = (0.5, 1.0, 0.0)
ENT = 0.01


class _Case:
    """nets, rollout, normalised returns and the update object of one pair on one batch.  Samples whose float64 ratio lies
    within 1e-4 of a clip edge, or whose relu input lies within 1e-4 of 0, get R_hat = V (so adv = 0 exactly): float32
    rounding may put them on the other side of the kink."""

    def __init__(self, pair, batch):
        from reinforcementlearningplatform_b200 import _lib as L
        from reinforcementlearningplatform_b200.learn import FusedPPO2Update
        actor_dims, critic_dims, head, std_vector = PAIRS[pair]
        kind, T, N, first, count = BATCHES[batch]
        S, A = actor_dims[0], actor_dims[-1]
        self.first, self.count, self.head, self.A = first, count, head, A
        seed = 100 * list(PAIRS).index(pair) + list(BATCHES).index(batch)
        torch.manual_seed(seed)
        self.a_min, self.a_max = -1.0 - 0.25 * np.arange(A), 2.0 + 0.5 * np.arange(A)
        off = (self.a_min + self.a_max) / 2
        self.std = np.linspace(0.3, 0.6, A) if std_vector else 0.45
        actor = _Net(actor_dims, head, self.a_max - off, off).to("cuda")
        critic = _Net(critic_dims).to("cuda")
        with torch.no_grad():
            actor[-1].weight.mul_(10.0 if head == "relu" else 3.0)
            if head == "relu":
                actor(torch.rand(4096, S, device="cuda") * 2 - 1)
                actor[-1].bias.sub_(actor.Z[-1].median(0).values)
        self.nets64 = copy.deepcopy(actor).double(), copy.deepcopy(critic).double()
        g = torch.Generator(device="cuda").manual_seed(seed)
        self.s = (torch.rand(T, S, N, device="cuda", generator=g) * 2 - 1).contiguous()
        sd = torch.as_tensor(self.std, dtype=torch.float32, device="cuda").reshape(-1).expand(A)
        with torch.no_grad():
            mean = actor(self.s.permute(0, 2, 1).reshape(T * N, S))
            af = mean + sd * torch.randn(mean.shape, device="cuda", generator=g)
            lp = -((af - mean) ** 2) / (2 * sd * sd) - torch.log(sd) - math.log(math.sqrt(2 * math.pi))
            lp = lp + (0.25 / math.sqrt(A)) * torch.randn(lp.shape, device="cuda", generator=g)
        self.a = af.reshape(T, N, A).permute(0, 2, 1).contiguous()
        self.a_lp = lp.reshape(T, N, A).permute(0, 2, 1).contiguous()
        self.ret_hat = torch.randn(T, N, device="cuda", generator=g).contiguous()
        B = T * N
        self.perm_key, self.index = 0, None
        if kind == "perm":
            self.perm_key = 4242 + seed
            out = np.empty(count, dtype=np.int64)
            L.check(L.load().b200_ppo2_permutation(self.perm_key, B, first, count, out.ctypes.data_as(C.POINTER(C.c_int64))),
                    "perm")
            self.sel = torch.as_tensor(out, device="cuda")
        else:
            pick = torch.randperm(B, device="cuda", generator=g)
            sel = pick[:count]
            if kind == "repeat":
                sel = torch.cat([pick[:count - count // 3], pick[:count // 3]])
                sel = sel[torch.randperm(count, device="cuda", generator=g)]
            self.sel = sel
            self.index = torch.cat([pick[-first:], sel, pick[-9:]]).contiguous()
        self.upd = FusedPPO2Update(actor, critic, self.std, self.a_min, self.a_max, head, entropy_coef=ENT)
        # kinks -> R_hat = V at those samples
        _, _, _, value = self.ppo1(0.5)
        t = self.terms()
        with torch.no_grad():
            near = lambda x, e: (x - e).abs() <= 1e-4 * e
            kink = near(t["ratio"], 0.8) | near(t["ratio"], 1.2)
            if head == "relu":
                kink |= (self.nets64[0].Z[-1][:, :A].abs() <= 1e-4).any(1)
        self.n_kink = int(kink.sum())
        self.ret_hat.view(-1)[self.sel[kink]] = value.view(-1)[self.sel[kink]]

    def ppo1(self, value_coef):
        """b200_ppo1_grad: ([actor grad, critic grad], losses, adv, value)"""
        adv = torch.full_like(self.ret_hat, float("nan"))
        value = torch.zeros_like(self.ret_hat)
        self.upd.ppo1_grad_step(self.s, self.a, self.a_lp, self.ret_hat, adv, value_coef, self.first, self.count,
                                perm_key=self.perm_key, index=self.index, value=value)
        o = self.upd.params.net_off[1]
        return [self.upd.grad[:o].clone(), self.upd.grad[o:].clone()], self.upd.loss.clone(), adv, value

    def ppo2(self, adv, v_target):
        self.upd.grad_step(self.s, self.a, self.a_lp, adv, v_target, self.first, self.count, perm_key=self.perm_key,
                           index=self.index)
        o = self.upd.params.net_off[1]
        return [self.upd.grad[:o].clone(), self.upd.grad[o:].clone()], self.upd.loss.clone()

    def flat(self, x):
        T, _, N = self.s.shape
        return x.permute(0, 2, 1).reshape(T * N, -1)[self.sel]

    def terms(self, adv=None):
        """float64 forward of both nets on the batch; with `adv` (the kernel's float32 advantage) also the backward of
        the joint loss with value_coef 1: the actor's surrogate and the critic's mse"""
        actor, critic = self.nets64
        for net in self.nets64:
            for p in net.parameters():
                p.grad = None
        sb, ab, lpb = (self.flat(x).double() for x in (self.s, self.a, self.a_lp))
        rh = self.ret_hat.reshape(-1, 1)[self.sel].double()
        mean = actor(sb)
        sd = torch.as_tensor(self.std, device="cuda", dtype=torch.float32).reshape(-1).double().expand(ab.shape[1])
        lp = -((ab - mean) ** 2) / (2 * sd * sd) - torch.log(sd) - math.log(math.sqrt(2 * math.pi))
        ent = (0.5 + 0.5 * math.log(2 * math.pi) + torch.log(sd)).sum()
        ratios = torch.exp(lp.sum(1, keepdim=True) - lpb.sum(1, keepdim=True))
        value = critic(sb)
        t = {"ratio": ratios.detach().reshape(-1), "value": value.detach().reshape(-1)}
        if adv is None:
            return t
        advb = adv.reshape(-1, 1)[self.sel].double()
        surr1, surr2 = ratios * advb, torch.clamp(ratios, 0.8, 1.2) * advb
        actor_loss = (-torch.min(surr1, surr2) - ENT * ent).mean()
        mse = ((value - rh) ** 2).mean()
        (actor_loss + mse).backward()
        clamped = (ratios < 0.8) | (ratios > 1.2)
        c = torch.where(clamped & ~(surr1 < surr2), 0.0, -advb) * ratios / len(self.sel)
        lp_abs = (((ab - mean) ** 2) / (2 * sd * sd) + torch.log(sd).abs() + math.log(math.sqrt(2 * math.pi))).sum(1) \
            + lpb.abs().sum(1)
        t.update(c=c.detach(), act=ab, mean=mean.detach(), var=sd * sd, lp_abs=lp_abs.detach().reshape(-1, 1))
        t["grads"] = [_flat_grads(actor), _flat_grads(critic)]
        t["scales"] = [_grad_scales(actor, _out_scale(actor, t)), _grad_scales(critic, critic.Z[-1].grad.abs())]
        surr = torch.min(surr1, surr2).detach().reshape(-1)
        t["losses"] = [float(actor_loss), float(mse)]
        t["lscales"] = [float((surr.abs() * (1 + lp_abs.detach())).mean()) + abs(ENT * float(ent)),
                        float(((value - rh) ** 2).detach().mean())]
        return t


_CACHE = {}


def _case(pair, batch):
    if (pair, batch) not in _CACHE:
        _CACHE.clear()
        _CACHE[(pair, batch)] = _Case(pair, batch)
    return _CACHE[(pair, batch)]


@pytest.mark.parametrize("pair,batch", CASES, ids=[f"{p}-{b}" for p, b in CASES])
def test_advantage_launch_is_the_critic_forward_of_the_grad_kernel(pair, batch):
    L = _lib()
    cs = _case(pair, batch)
    _, _, adv, value = cs.ppo1(0.5)
    sel = cs.sel
    # adv = R_hat - V, one float32 subtraction, at the batch's samples only
    assert torch.equal(adv.view(-1)[sel], cs.ret_hat.view(-1)[sel] - value.view(-1)[sel])
    untouched = torch.ones(adv.numel(), dtype=torch.bool, device="cuda")
    untouched[sel] = False
    assert bool(torch.isnan(adv.view(-1)[untouched]).all())
    # a critic-only b200_ppo2_grad with v_target := V: every squared error is exactly 0 -> gradient and loss exactly 0
    upd, lib = cs.upd, L.load()
    b = upd._batch(cs.s, cs.a, cs.a_lp, adv, value, cs.first, cs.count, cs.perm_key, cs.index)
    cm = upd.params.mlp(1, 0)
    grad = torch.full((upd.params.net_len[1],), float("nan"), device="cuda")
    loss = torch.full((2,), float("nan"), device="cuda")
    L.check(lib.b200_ppo2_grad(C.byref(b), None, C.byref(cm), upd.std, _p(upd.std_vec), _p(upd.a_min), _p(upd.a_max),
                               upd.eps_clip, upd.entropy_coef, None, _p(grad), _p(loss), _p(upd.workspace),
                               upd.workspace.numel(), _stream()), "b200_ppo2_grad")
    assert bool((grad == 0).all()) and float(loss[1]) == 0.0
    # V within K-LEARN's bound of a float64 forward
    t = cs.terms()
    _, zc = _fwd_scales(cs.nets64[1])
    worst = _ratio(value.view(-1)[sel].double() - t["value"], zc.reshape(-1))
    print(f"\n{pair}-{batch}: V within {worst:.2f} x 2^-24 scale of float64")
    assert worst <= C_GRAD, worst


@pytest.mark.parametrize("pair,batch", CASES, ids=[f"{p}-{b}" for p, b in CASES])
def test_exact_links_to_the_ppo2_path(pair, batch):
    cs = _case(pair, batch)
    g05, l05, adv, value = cs.ppo1(0.5)
    g1, l1, adv1, value1 = cs.ppo1(1.0)
    sel = cs.sel                              # adv / value are written at the batch's samples only
    assert torch.equal(adv1.view(-1)[sel], adv.view(-1)[sel]) and torch.equal(value1.view(-1)[sel], value.view(-1)[sel])
    gp, lp = cs.ppo2(adv, cs.ret_hat)         # PPO2 with adv from the advantage launch and v_target = R_hat
    # value_coef 0.5: exactly half of PPO2's critic gradient and loss; the actor's gradient is PPO2's
    assert torch.equal(g05[1], 0.5 * gp[1]) and float(l05[1]) == 0.5 * float(lp[1])
    assert torch.equal(g05[0], gp[0]) and float(l05[0]) == float(lp[0])
    # value_coef 1: the two-step PPO2 path
    assert all(torch.equal(x, y) for x, y in zip(g1, gp)) and torch.equal(l1, lp)
    # repeated launches give the same bits
    g05b, l05b, adv_b, _ = cs.ppo1(0.5)
    assert all(torch.equal(x, y) for x, y in zip(g05, g05b)) and torch.equal(l05, l05b)
    assert torch.equal(adv.view(-1)[sel], adv_b.view(-1)[sel])


@pytest.mark.parametrize("pair,batch", CASES, ids=[f"{p}-{b}" for p, b in CASES])
def test_joint_loss_matches_float64_autograd(pair, batch):
    cs = _case(pair, batch)
    assert cs.n_kink <= max(1, 0.01 * cs.count), cs.n_kink
    worst = {}
    for vc in VALUE_COEFS:
        grads, loss, adv, _ = cs.ppo1(vc)
        t = cs.terms(adv)
        for j, name in ((0, "actor"), (1, "critic")):
            k = 1.0 if j == 0 else vc
            worst[f"{name} grad vc={vc}"] = _ratio(grads[j].double() - k * t["grads"][j], k * t["scales"][j])
            worst[f"{name} loss vc={vc}"] = _ratio(torch.tensor(float(loss[j]) - k * t["losses"][j]),
                                                   torch.tensor(k * t["lscales"][j]))
        if vc == 0.0:
            assert bool((grads[1] == 0).all()) and float(loss[1]) == 0.0
    print(f"\n{pair}-{batch}: worst {max(worst.values()):.2f}  " + "  ".join(f"{k} {v:.2f}" for k, v in worst.items())
          + f"  neutralised {cs.n_kink}")
    for k, v in worst.items():
        assert v <= C_GRAD, (k, v)


# ------------------------------------------------------------------------------------------------ 5. VecPPO.learn()
def _agent(n_envs=4096, T=32, epochs=4, std=0.8, seed=3, module_seed=11, ppo_msg=None, env_offset=0, group=None,
           **kw):
    import reinforcementlearningplatform_b200 as rlp
    from reinforcementlearningplatform_b200.ppo import VecPPO
    from reinforcementlearningplatform_b200.ppo2 import reference_nets
    env = rlp.CartPoleAngleOnly(n_envs=n_envs, variant="ppo2", io_dtype=torch.float32, auto_reset=True, seed=seed,
                                env_index_offset=env_offset)
    torch.manual_seed(module_seed)
    actor, critic = reference_nets(env.state_dim, env.action_dim, "cuda", init_std=std, mean_act="identity")
    msg = {"buffer_size": T, "K_epochs": epochs}
    msg.update(ppo_msg or {})
    agent = VecPPO(env, actor, critic, msg, std=std, seed=seed, group=group, **kw)
    env.reset(True)
    return agent


def _torch_epoch(actor, critic, opt, s, a, a_lp, ret_hat, std, eps_clip=0.2, ent_coef=0.01, value_coef=0.5):
    """one v1 epoch in float32 torch: the joint loss of the module docstring, one Adam step over both nets"""
    v = critic(s)
    adv = (ret_hat - v).detach()
    mean = actor(s)
    sd = torch.as_tensor(std, dtype=torch.float32, device=s.device).reshape(-1).expand(a.shape[1])
    lp = -((a - mean) ** 2) / (2 * sd * sd) - torch.log(sd) - math.log(math.sqrt(2 * math.pi))
    ent = (0.5 + 0.5 * math.log(2 * math.pi) + torch.log(sd)).sum()
    ratio = torch.exp(lp.sum(1, keepdim=True) - a_lp.sum(1, keepdim=True))
    surr = torch.min(ratio * adv, torch.clamp(ratio, 1 - eps_clip, 1 + eps_clip) * adv)
    loss = (-surr).mean() + value_coef * ((v - ret_hat) ** 2).mean() - ent_coef * ent
    opt.zero_grad()
    loss.backward()
    opt.step()
    return adv


def _restated_inputs(agent):
    from reinforcementlearningplatform_b200 import gae
    buf = agent.buffer
    T, N = buf.batch_size, buf.n_envs
    R = gae.mc_returns(buf.r, buf.done, agent.gamma).double()
    ret_hat = ((R - R.mean()) / (R.std() + 1e-7)).float().reshape(T * N, 1)
    flat = lambda x: x.permute(0, 2, 1).reshape(T * N, -1)
    return flat(buf.s), flat(buf.a), flat(buf.a_lp), ret_hat


def test_vecppo_learn_matches_a_torch_restatement():
    """4096 x 32 CartPoleAngleOnly samples, 4 epochs: the parameters after every epoch within PARAM_TOL of float32
    torch on copies of the modules (torch.optim.Adam, two parameter groups, eps 1e-8, no clip)"""
    one = _agent(epochs=1)                    # learn() with K_epochs = 1 four times on the same rollout = 4 epochs
    four = _agent(epochs=4)
    actor_t, critic_t = copy.deepcopy(one.actor), copy.deepcopy(one.critic)
    opt = torch.optim.Adam([{"params": actor_t.parameters(), "lr": 1e-4}, {"params": critic_t.parameters(), "lr": 1e-3}],
                           eps=1e-8)
    one.collect()
    four.collect()
    assert torch.equal(one.buffer.r, four.buffer.r) and torch.equal(one.buffer.a_lp, four.buffer.a_lp)
    s, a, a_lp, ret_hat = _restated_inputs(one)
    worst = []
    for e in range(4):
        out = one.learn()
        adv_t = _torch_epoch(actor_t, critic_t, opt, s, a, a_lp, ret_hat, 0.8)
        assert all(np.isfinite(v) for v in out.values()) and out["loss"] == out["actor_loss"] + out["critic_loss"]
        if e == 0:   # the advantage the epoch used: R_hat - V of the critic before the step
            assert float((one._adv.reshape(-1, 1) - adv_t).abs().max()) <= 1e-5
        d = max(float((p.detach() - q.detach()).abs().max())
                for m, mt in ((one.actor, actor_t), (one.critic, critic_t)) for p, q in zip(m.parameters(), mt.parameters()))
        worst.append(d)
    print(f"\nVecPPO vs torch: max |param difference| after each epoch {worst}")
    assert max(worst) <= PARAM_TOL, worst
    four.learn()
    assert torch.equal(one.fused.params.flat, four.fused.params.flat)
    # two runs with the same seed give the same bits
    again = _agent(epochs=4)
    again.collect()
    again.learn()
    assert torch.equal(again.fused.params.flat, four.fused.params.flat)


def test_ret_norm_eps_reaches_the_normalisation():
    """rewards scaled to ~1e-7: R_hat with the 1e-7 of (std + eps) differs by ~10 % from R_hat without it"""
    agent = _agent(n_envs=1024, T=16, epochs=1, ppo_msg={"ret_norm_eps": 1e-7})
    agent.collect()
    agent.buffer.r.mul_(1e-7)
    critic0 = copy.deepcopy(agent.critic)
    s, _, _, ret_hat = _restated_inputs(agent)
    agent.learn()
    with torch.no_grad():
        expect = ret_hat - critic0(s)
    assert float((agent._adv.reshape(-1, 1) - expect).abs().max()) <= 1e-5 * float(expect.abs().max())


# ------------------------------------------------------------------------------------------------ 6. training
def _example(*args):
    sys.path.insert(0, os.path.join(ROOT, "examples"))
    import train_ppo2_vec as T
    return T.main(list(args))


def test_vecppo_learns_cartpole_angleonly():
    log = _example("--algo", "ppo", "--env", "cartpole_angleonly", "--envs", "4096", "--steps", "64", "--iters", "25",
                   "--epochs", "25")
    assert all(np.isfinite(r["actor_loss"]) and np.isfinite(r["critic_loss"]) for r in log)
    first = np.mean([r["done_rate"] for r in log[:3]])
    last = np.mean([r["done_rate"] for r in log[-3:]])
    ret_first = np.nanmean([r["mean_episode_return"] for r in log[:3]])
    ret_last = np.nanmean([r["mean_episode_return"] for r in log[-3:]])
    print(f"\ndone rate {first:.4f} -> {last:.4f}; mean episode return {ret_first:.2f} -> {ret_last:.2f}")
    assert last < first, (first, last)
    assert ret_last > ret_first, (ret_first, ret_last)


def test_vecppo_runs_uav_hover():
    log = _example("--algo", "ppo", "--env", "uav_hover", "--envs", "4096", "--steps", "64", "--iters", "5", "--epochs", "4")
    assert len(log) == 5
    assert all(np.isfinite(r["actor_loss"]) and np.isfinite(r["critic_loss"]) and np.isfinite(r["loss"]) for r in log)
    assert sum(r["episodes"] for r in log) > 0


# ------------------------------------------------------------------------------------------------ 7. set_action_std
def test_set_action_std():
    import reinforcementlearningplatform_b200 as rlp  # noqa: F401
    set_ = _agent(n_envs=2048, T=16, epochs=2, std=0.5)
    set_.set_action_std(0.3)
    built = _agent(n_envs=2048, T=16, epochs=2, std=0.3)
    set_.collect()
    built.collect()
    for k in ("s", "a", "a_lp", "r", "done"):
        assert torch.equal(getattr(set_.buffer, k), getattr(built.buffer, k)), k
    set_.learn()
    built.learn()
    assert torch.equal(set_.fused.params.flat, built.fused.params.flat)
    # a change mid-run: the next rollout's log-probs are those of the new std
    set_.set_action_std(0.45)
    set_.collect()
    s, a, a_lp, _ = _restated_inputs(set_)
    with torch.no_grad():
        mean = set_.actor(s)
    lp = -((a - mean) ** 2) / (2 * 0.45 ** 2) - math.log(0.45) - math.log(math.sqrt(2 * math.pi))
    assert torch.allclose(a_lp, lp, atol=3e-5)
    assert set_.fused.std == float(np.float32(0.45)) and set_.policy.std == float(np.float32(0.45))


# ------------------------------------------------------------------------------------------------ 8. two ranks
N_TOTAL = 2048


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK="0")
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    torch.cuda.set_device(0)
    dist.init_process_group("gloo")
    from reinforcementlearningplatform_b200 import dist as D
    n, off = D.shard(N_TOTAL, rank, world)
    agent = _agent(n_envs=n, T=16, epochs=2, env_offset=off)
    agent.collect()
    agent.learn()
    q.put((rank, n, off, agent._ret_stats.cpu().numpy(), agent.fused.params.flat.cpu()))
    dist.destroy_process_group()


def test_two_ranks_match_one():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted((q.get(timeout=300) for _ in procs), key=lambda x: x[0])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    (_, n0, o0, st0, p0), (_, n1, o1, st1, p1) = res
    assert (n0, o0, n1, o1) == (1024, 0, 1024, 1024)
    one = _agent(n_envs=N_TOTAL, T=16, epochs=2)
    one.collect()
    from reinforcementlearningplatform_b200 import gae
    R = gae.mc_returns(one.buffer.r, one.buffer.done, one.gamma)
    x = R.double().cpu().numpy().ravel()
    one.learn()
    st = one._ret_stats.cpu().numpy()
    for s in (st0, st1, st):
        assert s[2] == x.size
        for k, v in ((0, x), (1, x * x)):
            exact = float(v.astype(np.longdouble).sum())
            assert abs(s[k] - exact) <= x.size * ULP_SUM * float(np.abs(v).astype(np.longdouble).sum()), (k, s[k], exact)
    assert torch.equal(p0, p1)
    d = float((p0.cuda() - one.fused.params.flat).abs().max())
    print(f"\ntwo ranks vs one: max |param difference| {d:.3e}")
    assert d <= PARAM_TOL, d
