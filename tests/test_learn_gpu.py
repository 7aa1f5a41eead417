"""K-LEARN (csrc/learn.cu) against a float64 autograd restatement of the PPO2 update.

The reference update is Proximal_Policy_Optimization2.learn (algorithm/policy_base/Proximal_Policy_Optimization2.py:
102-131): ``_torch_losses`` restates those lines (the same restatement round 1's VecPPO2 used, checked then against the
reference learner) and serves as the checker; the product path is the C ABI (b200_ppo2_grad / b200_adam_step /
b200_ppo2_learn).

Gradients: every entry within ``C_GRAD * 2^-24 * scale`` of float64 autograd on the same float32 inputs, where the scale
is the condition number of the sum the kernel computes: ``G_l^T Hc_l`` for the weights of layer l and ``sum_s G_l[s]``
for its bias (H_l the layer's input, dZ_l the gradient of its pre-activation, Hc_l >= |H_l| and G_l >= |dZ_l| the same
passes in absolute value: ``_grad_scales``), ``sum_s |per-sample loss term| / count`` for the losses.  Samples on a
kink of the loss are neutralised first (``_Case``).  The sweep (``ROWS`` x ``CASES``) reaches every register tile,
padding and block split of the kernel;
``test_sweep_covers_every_kernel_branch`` (CPU) restates the host's plan and keeps it that way.  Clip + Adam are checked
against a float64 restatement of ``adam_kernel``, entry by entry, and against ``torch.optim.Adam`` over several steps."""
import copy
import ctypes as C
import math

import numpy as np
import pytest
import torch

EPS32 = 2.0 ** -24
# 10x the largest ratio |g - g64| / (2^-24 scale) measured over the sweep (4.22 on a B200: the critic loss of the largest
# pair over 2^19 samples; DESIGN 4(c)); the ceiling is about the deepest summation the kernel does: 64 samples of a
# tile + tiles of a block + blocks of the reduction
C_GRAD = 48.0
C_CEILING = 256.0
# clip + Adam, in units of 2^-24: param within C_ADAM_P (|param_old| + |update|), m and v within C_ADAM_MV (|old| + |what
# the step adds|), the gradient norm within C_NORM |norm|.  Measured on a B200: 8.0, 1.0, 1.6
C_ADAM_P, C_ADAM_MV, C_NORM = 16.0, 4.0, 16.0

# actor dims, critic dims, actor head, per-dimension std vector, entropy_coef.  Register tiles (RN, RK) of fill_net in the
# comments; the CPU test below derives them and checks what the table covers.
ROWS = {
    "ref_relu": ((6, 64, 64, 32, 8), (6, 64, 32, 1), "relu", False, 0.01),          # (1,2) (4,4) (2,4) (1,1)
    "ref_identity": ((6, 64, 64, 32, 8), (6, 64, 32, 1), "identity", False, 0.01),
    "dppo2_64": ((41, 64, 64, 2), (41, 64, 64, 1), "tanh_range", True, 0.01),       # input padded 41 -> 48
    "w16": ((4, 16, 16, 1), (4, 16, 16, 1), "identity", False, 0.0),               # fwd_layer<2>, bwd_layer K = 16
    "w8": ((3, 8, 8, 2), (3, 8, 1), "relu", False, 0.01),                           # bwd_layer K = 8
    "a16": ((64, 32, 32, 16, 16), (64, 32, 32, 16, 1), "relu", True, 0.01),         # (1,4); 16 actions
    "two_layer": ((9, 64, 9), (9, 48, 1), "tanh_range", False, 0.01),               # (1,4) twice; 48 padded to 64
    "w20": ((5, 20, 3), (5, 20, 1), "identity", False, 0.01),                       # 20 padded to 32
    "one_layer": ((5, 3), (5, 1), "identity", False, 0.01),
    "s1": ((1, 64, 1), (1, 64, 1), "relu", False, 0.01),                            # input padded 1 -> 8
    "largest": ((64, 64, 64, 64, 16), (64, 64, 64, 64, 1), "relu", False, 0.01),    # ~129 KB of shared memory
}
# name -> (how the samples are picked, T, N, first, count).  "index": the `index` path at index[first:first + count] of a
# longer index tensor; "repeat": the same with repeated samples; "perm": the kernel's keyed permutation of the rollout
BATCHES = {
    "i1": ("index", 4, 1000, 17, 1),
    "i63": ("index", 4, 1000, 17, 63),
    "r65": ("repeat", 4, 1000, 17, 65),
    "i3001": ("index", 4, 1000, 17, 3001),
    "p16k": ("perm", 32, 1 << 14, 3 << 14, 1 << 14),
    "p64k": ("perm", 32, 1 << 14, 1 << 16, 1 << 16),
    "p512k": ("perm", 32, 1 << 14, 0, 1 << 19),          # the whole rollout as one mini-batch
    "n1": ("perm", 6000, 1, 0, 6000),                     # one environment, a long rollout
    "t1": ("perm", 1, 5000, 100, 4000),                   # one step of many environments
}
# the DPPO2 demo head (tanh range, per-dimension std) runs in test_tanh_range_head_with_std_vector, every other row here
TANH_RANGE_CASES = [("dppo2_64", b) for b in ("i1", "i63", "r65", "i3001", "p64k")]
CASES = [(r, b) for r in ROWS if r != "dppo2_64" for b in ("i1", "i63", "r65", "i3001")] + [
    ("ref_relu", "p16k"), ("ref_relu", "p64k"), ("ref_relu", "p512k"),
    ("largest", "p16k"), ("largest", "p64k"), ("largest", "p512k"),
    ("a16", "p16k"), ("ref_identity", "n1"), ("w8", "t1")]
SINGLE_NET_CASES = [("ref_relu", "p64k"), ("two_layer", "i3001")]
GRID_CAP = 296   # 148 SMs x 2 blocks (learn.cu: GRID_CAP, grid_cap())


# ------------------------------------------------------------------------------------------------ host plan (CPU)
def _plan(dims):
    """fill_net: per layer (K, N, (RN, RK)) -- K the padded input width, N the padded output width, (RN, RK) the
    register tile of the weight-gradient product"""
    out = []
    for l, (i, o) in enumerate(zip(dims[:-1], dims[1:])):
        K = (i + 7) // 8 * 8 if l == 0 else out[-1][1]
        N = 8 if o <= 8 else 16 if o <= 16 else 32 if o <= 32 else 64
        e = 1
        while e < 16 and N * K > e * 256:
            e *= 2
        out.append((K, N, (e // min(e, 4), min(e, 4))))
    return out


def _split(nets, count):
    """launch_grad: (blocks, most tiles per block) of each net in the launch"""
    tiles = -(-count // 64)
    if len(nets) == 1:
        nblk = [min(tiles, GRID_CAP)]
    else:
        w = [sum(K * N for K, N, _ in _plan(d)) + 2200.0 for d in nets]
        nb1 = min(GRID_CAP - 1, max(1, int(GRID_CAP * w[1] / (w[0] + w[1]) + 0.5)))
        nblk = [min(tiles, GRID_CAP - nb1), min(tiles, nb1)]
    return [(n, -(-tiles // n)) for n in nblk]


def test_sweep_covers_every_kernel_branch():
    tiles, nj, bwd_k, depths, acts, per_block, reduce_wide = set(), set(), set(), set(), set(), set(), set()
    launches = [((ROWS[r][0], ROWS[r][1]), b) for r, b in CASES + TANH_RANGE_CASES]
    launches += [((ROWS[r][k],), b) for r, b in SINGLE_NET_CASES for k in (0, 1)]
    for nets, b in launches:
        for dims in nets:
            p = _plan(dims)
            depths.add(len(p))
            for l, (K, N, t) in enumerate(p):
                tiles.add(t)
                nj.add(N // 8)
                if l > 0:
                    bwd_k.add(K)
        A = nets[0][-1]
        acts.add("1" if A == 1 else "<=8" if A <= 8 else ">8")
        for nblk, most in _split(nets, BATCHES[b][4]):
            per_block.add(most > 1)
            reduce_wide.add(nblk >= 8)
    assert tiles == {(4, 4), (2, 4), (1, 4), (1, 2), (1, 1)}
    assert nj == {1, 2, 4, 8} and bwd_k == {8, 16, 32, 64} and depths == {1, 2, 3, 4}
    assert acts == {"1", "<=8", ">8"}
    assert per_block == {False, True} and reduce_wide == {False, True}
    # the whole-rollout case keeps >= 40 tiles in every block
    assert min(m for _, m in _split(ROWS["ref_relu"][:2], BATCHES["p512k"][4])) >= 40
    assert C_GRAD <= C_CEILING


# ------------------------------------------------------------------------------------------------ references
def _rollout(T, S, A, N, seed, a_lo=0.0, a_hi=5.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    r = lambda *shape: torch.rand(*shape, device="cuda", generator=g)
    s = (r(T, S, N) * 2 - 1).contiguous()
    a = (a_lo + (a_hi - a_lo) * r(T, A, N)).contiguous()
    a_lp = (-1.5 - 0.5 * r(T, A, N)).contiguous()
    adv = torch.randn(T, N, device="cuda", generator=g).contiguous()
    vt = (3 * torch.randn(T, N, device="cuda", generator=g)).contiguous()
    return s, a, a_lp, adv, vt


def _torch_losses(actor, critic, std, s, a, a_lp, adv, vt, idx, eps_clip=0.2, ent_coef=0.01, dtype=None, terms=None):
    """PPO2.py:106-124 on the flat batch picked by idx (positions b = t * N + i).  ``terms``: a dict that receives the
    per-sample ratio, advantage, min(surr1, surr2) and squared value error, and the entropy."""
    T, S, N = s.shape
    flat = lambda x: x.permute(0, 2, 1).reshape(T * N, -1)
    cast = (lambda x: x.to(dtype)) if dtype is not None else (lambda x: x)
    sb, ab, lpb = cast(flat(s)[idx]), cast(flat(a)[idx]), cast(flat(a_lp)[idx])
    advb, vtb = cast(adv.reshape(-1, 1)[idx]), cast(vt.reshape(-1, 1)[idx])
    mean = actor(sb)
    sd = cast(torch.as_tensor(std, device=s.device, dtype=torch.float32).reshape(-1)).expand(ab.shape[1])
    lp = -((ab - mean) ** 2) / (2 * sd * sd) - torch.log(sd) - math.log(math.sqrt(2 * math.pi))
    ent = (0.5 + 0.5 * math.log(2 * math.pi) + torch.log(sd)).sum()
    ratios = torch.exp(lp.sum(1, keepdim=True) - lpb.sum(1, keepdim=True))
    surr1 = ratios * advb
    surr2 = torch.clamp(ratios, 1 - eps_clip, 1 + eps_clip) * advb
    actor_loss = (-torch.min(surr1, surr2) - ent_coef * ent).mean()
    value = critic(sb)
    critic_loss = torch.nn.functional.mse_loss(vtb, value)
    if terms is not None:
        # c: d actor_loss / d lp of each sample (0 where the clamp is active and selected)
        clamped = (ratios < 1 - eps_clip) | (ratios > 1 + eps_clip)
        c = torch.where(clamped & ~(surr1 < surr2), 0.0, -advb) * ratios / len(idx)
        lp_abs = (((ab - mean) ** 2) / (2 * sd * sd) + torch.log(sd).abs() + math.log(math.sqrt(2 * math.pi))).sum(1) + lpb.abs().sum(1)
        terms.update(ratio=ratios.detach().reshape(-1), adv=advb.reshape(-1), surr=torch.min(surr1, surr2).detach().reshape(-1),
                     sq=((vtb - value) ** 2).detach().reshape(-1), ent=float(ent), c=c.detach(), act=ab, mean=mean.detach(),
                     var=sd * sd, lp_abs=lp_abs.detach().reshape(-1, 1))
    return actor_loss, critic_loss


def _flat_grads(actor, critic):
    from reinforcementlearningplatform_b200.policy import linear_layers
    out = []
    for net in (actor, critic):
        out.append(torch.cat([p.grad.reshape(-1) for lin in linear_layers(net) for p in (lin.weight, lin.bias)]))
    return out


class _Net(torch.nn.Sequential):
    """nn.Linear layers, tanh between them, ``head`` on the last (identity / relu / tanh_range = tanh(z) gain + off).
    forward() keeps every layer's input H_l and pre-activation Z_l (the output's gradient retained) for the
    error bound."""

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


def _grad_scales(net, g_out):
    """per flat gradient entry, layer by layer: G_l^T Hc_l (weights) and sum_s G_l[s] (bias).  The kernel's sums are
    dW_l = dZ_l^T H_l and db_l = sum_s dZ_l, but dZ_l and H_l are themselves rounded results, so both factors are
    replaced by what the passes give with every product and sum taken in absolute value:
        forward   Hc_0 = |x|,  Hc_{l+1} = |H_{l+1}| + (1 - H_{l+1}^2) (Hc_l |W_l|^T + |b_l|)
        backward  G_L = g_out (>= |dZ_L|: _out_scale),  G_{l-1} = (G_l |W_l|) * (1 - H_l^2)
    (Hc_l >= |H_l|, G_l >= |dZ_l|.)  With |H_l|, |dZ_l| alone, an activation near 0 or a cancelling sum dZ_l W_l puts
    float32 autograd itself 250x 2^-24 from float64 on a one-sample batch."""
    Hc = [net.H[0].abs()]
    for l in range(len(net) - 1):
        zc = Hc[l] @ net[l].weight.detach().abs().t() + net[l].bias.detach().abs()
        Hc.append(net.H[l + 1].abs() + (1 - net.H[l + 1] ** 2) * zc)
    G = g_out
    out = []
    for l in range(len(net) - 1, -1, -1):
        out = [(G.t() @ Hc[l]).reshape(-1), G.sum(0)] + out
        if l > 0:
            G = (G @ net[l].weight.detach().abs()) * (1 - net.H[l] ** 2)
    return torch.cat(out)


def _out_scale(actor, t):
    """G_L of the actor: dZ_L = c (act - m) / var * dm/dz, evaluated in absolute value.  The subtraction act - m cancels
    where an action was drawn close to the mean, and c carries the rounding of the log-prob sum inside the ratio
    (lp_abs: the sum of its terms in absolute value)."""
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


def _make(state_dim=6, action_dim=8, mean_act="relu", scale_mean=30.0, seed=0):
    from reinforcementlearningplatform_b200.ppo2 import reference_nets
    torch.manual_seed(seed)
    actor, critic = reference_nets(state_dim, action_dim, "cuda", init_std=0.45, mean_act=mean_act)
    with torch.no_grad():
        actor.mean_layer.weight.mul_(scale_mean)     # gain-0.01 init would leave the relu head almost flat
        actor.mean_layer.bias.add_(0.3)
    return actor, critic, copy.deepcopy(actor), copy.deepcopy(critic)


class _Case:
    """One row of ROWS on one batch of BATCHES: nets, rollout, the kernel's update object and the float64 / float32
    autograd references.  Samples whose float64 ratio lies within 1e-4 of a clip edge, or whose relu input lies within
    1e-4 of 0, get adv = 0: float32 rounding may put them on the other side of the kink, where the gradient jumps by a
    whole sample's contribution."""

    def __init__(self, row, batch, seed=0):
        from reinforcementlearningplatform_b200 import _lib
        from reinforcementlearningplatform_b200.learn import FusedPPO2Update
        actor_dims, critic_dims, head, std_vector, ent = ROWS[row]
        kind, T, N, first, count = BATCHES[batch]
        S, A = actor_dims[0], actor_dims[-1]
        self.row, self.batch, self.first, self.count, self.ent = row, batch, first, count, ent
        self.head, self.A = head, A
        seed = seed + 1000 * list(ROWS).index(row) + list(BATCHES).index(batch)
        torch.manual_seed(seed)
        self.a_min, self.a_max = -1.0 - 0.25 * np.arange(A), 2.0 + 0.5 * np.arange(A)   # (lo + hi) / 2 exact in float32
        off = (self.a_min + self.a_max) / 2
        self.std = np.linspace(0.3, 0.6, A) if std_vector else 0.45
        actor = _Net(actor_dims, head, self.a_max - off, off).to("cuda")
        critic = _Net(critic_dims).to("cuda")
        with torch.no_grad():
            # a head with spread: both sides of relu, of the clip range, of tanh's knee
            actor[-1].weight.mul_(10.0 if head == "relu" else 3.0)
            if head == "relu":                # about half of the relu outputs dead
                actor(torch.rand(4096, S, device="cuda") * 2 - 1)
                actor[-1].bias.sub_(actor.Z[-1].median(0).values)
        self.nets64 = copy.deepcopy(actor).double(), copy.deepcopy(critic).double()
        self.nets32 = copy.deepcopy(actor), copy.deepcopy(critic)

        g = torch.Generator(device="cuda").manual_seed(seed)
        s = (torch.rand(T, S, N, device="cuda", generator=g) * 2 - 1).contiguous()
        sd = torch.as_tensor(self.std, dtype=torch.float32, device="cuda").reshape(-1).expand(A)
        with torch.no_grad():
            # actions as choose_action draws them (PPO2.py:72-75) and log-probs of a slightly older policy: the ratios
            # straddle the clip range
            mean = actor(s.permute(0, 2, 1).reshape(T * N, S))
            af = mean + sd * torch.randn(mean.shape, device="cuda", generator=g)
            lp = -((af - mean) ** 2) / (2 * sd * sd) - torch.log(sd) - math.log(math.sqrt(2 * math.pi))
            lp = lp + (0.25 / math.sqrt(A)) * torch.randn(lp.shape, device="cuda", generator=g)
        self.s = s
        self.a = af.reshape(T, N, A).permute(0, 2, 1).contiguous()
        self.a_lp = lp.reshape(T, N, A).permute(0, 2, 1).contiguous()
        self.adv = torch.randn(T, N, device="cuda", generator=g).contiguous()
        self.vt = (3 * torch.randn(T, N, device="cuda", generator=g)).contiguous()

        B = T * N
        self.perm_key, self.index = 0, None
        if kind == "perm":
            self.perm_key = 4242 + seed
            out = np.empty(count, dtype=np.int64)
            _lib.check(_lib.load().b200_ppo2_permutation(self.perm_key, B, first, count,
                                                          out.ctypes.data_as(C.POINTER(C.c_int64))), "perm")
            self.sel = torch.as_tensor(out, device="cuda")
        else:
            pick = torch.randperm(B, device="cuda", generator=g)
            if kind == "repeat":
                sel = torch.cat([pick[:count - count // 3], pick[:count // 3]])
                sel = sel[torch.randperm(count, device="cuda", generator=g)]
            else:
                sel = pick[:count]
            self.sel = sel
            self.index = torch.cat([pick[-first:], sel, pick[-9:]]).contiguous()   # first != 0, a tail after the batch
        assert torch.equal(self.index[first:first + count], self.sel) if self.index is not None else True

        # kinks -> adv = 0 (float64 forward on the exact float32 inputs)
        t = {}
        with torch.no_grad():
            _torch_losses(*self.nets64, self.std, s, self.a, self.a_lp, self.adv, self.vt, self.sel, ent_coef=ent,
                          dtype=torch.float64, terms=t)
            near = lambda x, e: (x - e).abs() <= 1e-4 * e
            kink = near(t["ratio"], 0.8) | near(t["ratio"], 1.2)
            if head == "relu":
                kink |= (self.nets64[0].Z[-1][:, :A].abs() <= 1e-4).any(1)
        self.n_kink = int(kink.sum())
        self.adv.view(-1)[self.sel[kink]] = 0.0

        self.upd = FusedPPO2Update(actor, critic, self.std, self.a_min, self.a_max, head, entropy_coef=ent)

    def rollout(self):
        return self.s, self.a, self.a_lp, self.adv, self.vt

    def run(self):
        """the kernel: ([actor grad, critic grad], [actor loss, critic loss])"""
        self.upd.grad_step(*self.rollout(), self.first, self.count, perm_key=self.perm_key, index=self.index)
        o = self.upd.params.net_off[1]
        return [self.upd.grad[:o].clone(), self.upd.grad[o:].clone()], self.upd.loss.clone()

    def reference(self, nets, dtype=None):
        """autograd on `nets`: (flat grads, losses, per-entry grad scales, loss scales, per-sample terms)"""
        for net in nets:
            for p in net.parameters():
                p.grad = None
        t = {}
        la, lc = _torch_losses(*nets, self.std, *self.rollout(), self.sel, ent_coef=self.ent, dtype=dtype, terms=t)
        la.backward()
        lc.backward()
        grads = _flat_grads(*nets)
        scales = [_grad_scales(nets[0], _out_scale(nets[0], t)), _grad_scales(nets[1], nets[1].Z[-1].grad.abs())]
        lscale = [float((t["surr"].abs() * (1 + t["lp_abs"].reshape(-1))).mean()) + abs(self.ent * t["ent"]),
                  float(t["sq"].mean())]
        return grads, [float(la), float(lc)], scales, lscale, t


# ------------------------------------------------------------------------------------------------ the sweep
def _bound_ratios(name, grads, losses, ref, which=(0, 1)):
    """largest |kernel - f64| / (2^-24 scale) over the gradient entries and the loss of each net in `which`"""
    g64, l64, scales, lscale, _ = ref
    worst = {}
    for j in which:
        worst[f"{'actor' if j == 0 else 'critic'} grad"] = _ratio(grads[j].double() - g64[j], scales[j])
        worst[f"{'actor' if j == 0 else 'critic'} loss"] = _ratio(torch.tensor(losses[j] - l64[j]),
                                                                   torch.tensor(lscale[j]))
    return worst


def _check_case(row, batch):
    """one case of the sweep: the kernel's gradients and losses within the float64-derived bound, the old float32
    autograd comparison, what the case exercises, and bit-identical repeated launches"""
    cs = _Case(row, batch)
    grads, loss = cs.run()
    ref = cs.reference(cs.nets64, torch.float64)
    g64, l64, scales, lscale, t = ref
    g32, l32, _, _, _ = cs.reference(cs.nets32)
    mine = _bound_ratios("kernel", grads, loss.tolist(), ref)
    torch32 = _bound_ratios("torch", [g.double() for g in g32], l32, ref)
    print(f"\n{row}-{batch}: C kernel {max(mine.values()):.2f} torch-f32 {max(torch32.values()):.2f}  "
          + "  ".join(f"{k} {v:.2f}/{torch32[k]:.2f}" for k, v in mine.items()) + f"  neutralised {cs.n_kink}")
    for k, v in mine.items():
        assert v <= C_GRAD, (k, v, mine)
    for j in (0, 1):   # within 1e-6 of float32 autograd, or as close to float64 as float32 autograd itself (x2)
        err, err32 = float((grads[j].double() - g64[j]).abs().max()), float((g32[j].double() - g64[j]).abs().max())
        assert float((grads[j] - g32[j]).abs().max()) <= 1e-6 or err <= max(2e-6 * float(g64[j].abs().max()), 2 * err32)
    assert cs.n_kink <= max(1, 0.01 * cs.count), cs.n_kink

    if cs.count >= 3001:
        assert all(float(s.max()) > 0 for s in scales)
        # the case exercises both branches of the clipped surrogate, both signs of adv and (relu) both sides of the head
        clamped = (t["ratio"] < 0.8) | (t["ratio"] > 1.2)
        selected = clamped & ~(t["ratio"] * t["adv"] < torch.clamp(t["ratio"], 0.8, 1.2) * t["adv"])
        share = float(selected.double().mean())
        assert 0.05 <= share <= 0.95, share
        assert bool((t["adv"] > 0).any()) and bool((t["adv"] < 0).any())
        if cs.head == "relu":
            dead = float((cs.nets64[0].Z[-1][:, :cs.A] <= 0).double().mean())
            assert 0.05 <= dead <= 0.95, dead

    # bit-reproducible: no atomics, the per-block partials summed in block order
    grads2, loss2 = cs.run()
    assert all(torch.equal(a, b) for a, b in zip(grads, grads2)) and torch.equal(loss, loss2)


@pytest.mark.gpu
@pytest.mark.parametrize("row,batch", CASES, ids=[f"{r}-{b}" for r, b in CASES])
def test_gradients_match_autograd(row, batch):
    _check_case(row, batch)


@pytest.mark.gpu
def test_tanh_range_head_with_std_vector():
    """the DPPO2 demos' actor head (mean = tanh(z) * gain + off, per-dimension std) on a net K-LEARN can hold, on every
    batch shape of its row"""
    for row, batch in TANH_RANGE_CASES:
        _check_case(row, batch)


@pytest.mark.gpu
@pytest.mark.parametrize("row,batch", SINGLE_NET_CASES, ids=[f"{r}-{b}" for r, b in SINGLE_NET_CASES])
def test_single_net_launches(row, batch):
    """b200_ppo2_grad with the critic NULL, then with the actor NULL: each gradient against float64, and the loss lands
    in the launched net's slot of loss_out (the other slot is left alone)"""
    from reinforcementlearningplatform_b200 import _lib
    cs = _Case(row, batch, seed=7)
    lib, upd = _lib.load(), cs.upd
    ref = cs.reference(cs.nets64, torch.float64)
    b = upd._batch(*cs.rollout(), cs.first, cs.count, cs.perm_key, cs.index)
    p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
    mlp = [upd.params.mlp(0, upd.out_act), upd.params.mlp(1, 0)]
    for j in (0, 1):
        grad = torch.full((upd.params.net_len[j],), float("nan"), device="cuda")
        loss = torch.full((2,), float("nan"), device="cuda")
        nets = [C.byref(mlp[0]) if j == 0 else None, C.byref(mlp[1]) if j == 1 else None]
        ws = int(lib.b200_ppo2_workspace_bytes(*nets))
        assert 0 < ws <= upd.workspace.numel()
        _lib.check(lib.b200_ppo2_grad(
            C.byref(b), *nets, upd.std, p(upd.std_vec), p(upd.a_min), p(upd.a_max), upd.eps_clip, upd.entropy_coef,
            p(grad) if j == 0 else None, p(grad) if j == 1 else None, p(loss), p(upd.workspace), ws,
            upd._stream()), "b200_ppo2_grad")
        losses = [float("nan")] * 2
        losses[j] = float(loss[j])
        grads = [None, None]
        grads[j] = grad
        worst = _bound_ratios("kernel", grads, losses, ref, which=(j,))
        print(f"\n{row}-{batch} net {j} alone: " + "  ".join(f"{k} {v:.2f}" for k, v in worst.items()))
        for k, v in worst.items():
            assert v <= C_GRAD, (k, v)
        assert math.isnan(float(loss[1 - j])), loss.tolist()


# ------------------------------------------------------------------------------------------------ clip + Adam
def _adam64(p, g, m, v, lr, step, b1, b2, eps, max_norm, gs):
    """adam_kernel in float64: clip_grad_norm_ (1e-6 guard) of grad * grad_scale, then torch.optim.Adam's step"""
    p, g, m, v = (x.double() for x in (p, g, m, v))
    norm = float((g * gs).norm())
    coef = gs * (min(max_norm / (norm + 1e-6), 1.0) if max_norm > 0 else 1.0)
    g = g * coef
    m = m + (g - m) * (1 - b1)
    v = v * b2 + (1 - b2) * g * g
    delta = lr / (1 - b1 ** step) * m / (v.sqrt() / math.sqrt(1 - b2 ** step) + eps)
    return p - delta, m, v, norm, delta, g


@pytest.mark.gpu
@pytest.mark.parametrize("clip", ["off", "inactive", "active"])
@pytest.mark.parametrize("lens", [(1,), (1000,), (17153,), (300000,), (1, 300000), (17153, 1000)],
                         ids=lambda x: "-".join(map(str, x)))
def test_adam_step_matches_float64(lens, clip):
    from reinforcementlearningplatform_b200 import _lib
    lib = _lib.load()
    f32 = lambda x: float(np.float32(x))
    b1, b2, eps = f32(0.9), f32(0.999), f32(1e-5)
    lr = [f32(1e-3), f32(3e-4)][:len(lens)]
    offs, o = [], 3
    for n in lens:                   # segments with gaps: entries outside them must stay untouched
        offs.append(o)
        o += n + 5
    g = torch.Generator(device="cuda").manual_seed(sum(lens) + len(lens))
    P = o
    p0 = torch.randn(P, device="cuda", generator=g)
    g0 = torch.randn(P, device="cuda", generator=g) * 1e-2
    m0 = torch.randn(P, device="cuda", generator=g) * 1e-3
    v0 = torch.rand(P, device="cuda", generator=g) * 1e-5
    inside = torch.zeros(P, dtype=torch.bool, device="cuda")
    for so, n in zip(offs, lens):
        inside[so:so + n] = True
    worst = {"param": 0.0, "m": 0.0, "v": 0.0, "norm": 0.0}
    for step in (1, 7, 10 ** 4):
        for gs in (1.0, 0.125):
            norms = [float((g0[so:so + n].double() * gs).norm()) for so, n in zip(offs, lens)]
            max_norm = {"off": 0.0, "inactive": 2 * max(norms), "active": 0.5 * min(norms)}[clip]
            max_norm = f32(max_norm)
            p, m, v = p0.clone(), m0.clone(), v0.clone()
            norm_out = torch.full((2,), float("nan"), device="cuda")
            _lib.check(lib.b200_adam_step(
                len(lens), (C.c_int64 * 2)(*offs), (C.c_int64 * 2)(*lens), (C.c_float * 2)(*lr), C.c_void_p(p.data_ptr()),
                C.c_void_p(g0.data_ptr()), C.c_void_p(m.data_ptr()), C.c_void_p(v.data_ptr()), step, b1, b2, eps, max_norm,
                gs, C.c_void_p(norm_out.data_ptr()), C.c_void_p(torch.cuda.current_stream().cuda_stream)), "adam")
            for x, x0 in ((p, p0), (m, m0), (v, v0)):
                assert torch.equal(x[~inside], x0[~inside])
            for k, (so, n) in enumerate(zip(offs, lens)):
                sl = slice(so, so + n)
                p64, m64, v64, n64, d64, gc64 = _adam64(p0[sl], g0[sl], m0[sl], v0[sl], lr[k], step, b1, b2, eps,
                                                        max_norm, gs)
                assert n64 == pytest.approx(norms[k], rel=1e-12)
                r = {"param": _ratio(p[sl].double() - p64, p0[sl].double().abs() + d64.abs()),
                     "m": _ratio(m[sl].double() - m64, m0[sl].double().abs() + gc64.abs()),
                     "v": _ratio(v[sl].double() - v64, v0[sl].double().abs() + gc64 * gc64),
                     "norm": abs(float(norm_out[k]) - n64) / (EPS32 * n64)}
                for key in worst:
                    worst[key] = max(worst[key], r[key])
            if clip == "active":
                assert all(n > max_norm for n in norms)
    print(f"\nadam {lens} clip {clip}: ulp ratios " + "  ".join(f"{k} {v:.2f}" for k, v in worst.items()))
    assert worst["param"] <= C_ADAM_P and worst["m"] <= C_ADAM_MV and worst["v"] <= C_ADAM_MV, worst
    assert worst["norm"] <= C_NORM, worst


@pytest.mark.gpu
def test_clip_and_adam_match_torch_over_several_steps():
    from reinforcementlearningplatform_b200.learn import FusedPPO2Update
    actor, critic, actor_t, critic_t = _make()
    T, S, A, N = 4, 6, 8, 1024
    s, a, a_lp, adv, vt = _rollout(T, S, A, N, 2)
    vt = (vt * 10).contiguous()                     # large value targets: the critic's gradient norm exceeds the 0.5 clip
    upd = FusedPPO2Update(actor, critic, 0.45, np.zeros(A), np.full(A, 5.0), "relu", a_lr=1e-4, c_lr=1e-3, adam_eps=1e-5)
    oa = torch.optim.Adam(actor_t.parameters(), lr=1e-4, eps=1e-5)
    oc = torch.optim.Adam(critic_t.parameters(), lr=1e-3, eps=1e-5)
    g = torch.Generator(device="cuda").manual_seed(5)
    for step in range(4):
        idx = torch.randperm(T * N, device="cuda", generator=g)[:2048]
        upd.grad_step(s, a, a_lp, adv, vt, 0, 2048, index=idx)
        upd.adam_step()
        la, lc = _torch_losses(actor_t, critic_t, 0.45, s, a, a_lp, adv, vt, idx)
        oa.zero_grad(); la.backward()
        na = torch.nn.utils.clip_grad_norm_(actor_t.parameters(), 0.5)
        oa.step()
        oc.zero_grad(); lc.backward()
        nc = torch.nn.utils.clip_grad_norm_(critic_t.parameters(), 0.5)
        oc.step()
        mine = upd.grad_norm.tolist()
        assert abs(mine[0] - float(na)) <= 1e-5 * max(1.0, float(na)) and abs(mine[1] - float(nc)) <= 1e-5 * max(1.0, float(nc))
        assert float(nc) > 0.5                      # the critic's gradient is actually clipped
        # |delta param| <= 1e-6 for the actor; for the critic (lr 1e-3, value targets x10) 2e-3 of one Adam step (whose
        # size is <= lr): where |g| ~ eps = 1e-5 the update lr g / (|g| + eps) turns a 1e-8 difference of float32
        # summation order into 2.5e-4 lr -- torch against torch with another reduction order differs as much
        for net, ref, tol in ((actor, actor_t, 1e-6), (critic, critic_t, 2e-6)):
            for p, q in zip(net.parameters(), ref.parameters()):
                assert float((p.detach() - q.detach()).abs().max()) <= tol, (step, float((p.detach() - q.detach()).abs().max()))


@pytest.mark.gpu
def test_keyed_permutation_visits_every_sample_once_and_loop_matches_steps():
    from reinforcementlearningplatform_b200.learn import FusedPPO2Update
    actor, critic, _, _ = _make(seed=3)
    T, S, A, N = 5, 6, 8, 333                       # B = 1665: not a power of two, not a multiple of the tile
    s, a, a_lp, adv, vt = _rollout(T, S, A, N, 3)
    B = T * N
    nets = {mn: (copy.deepcopy(actor), copy.deepcopy(critic)) for mn in (0.5, 0.0)}
    upd = FusedPPO2Update(actor, critic, 0.45, np.zeros(A), np.full(A, 5.0), "relu")
    upd.grad_step(s, a, a_lp, adv, vt, 0, B, index=torch.arange(B, device="cuda"))
    full = upd.grad.clone()
    acc = torch.zeros_like(full, dtype=torch.float64)
    per_mb = []
    for first in range(0, B, 400):
        cnt = min(400, B - first)
        upd.grad_step(s, a, a_lp, adv, vt, first, cnt, perm_key=77)
        acc += upd.grad.double() * cnt / B
        per_mb.append(upd.grad.clone())
    assert float((acc - full.double()).abs().max()) <= 3e-6 * float(full.abs().max())
    upd.grad_step(s, a, a_lp, adv, vt, 0, 400, perm_key=78)      # another key = another mini-batch
    assert float((upd.grad - per_mb[0]).abs().max()) > 1e-3 * float(full.abs().max())
    # b200_ppo2_learn (C loop) == the same sequence of grad_step / adam_step calls, with the gradient clip and without it
    # (max_grad_norm = 0, what VecPPO2 passes when use_grad_clip is off)
    for max_norm, (actor1, critic1) in nets.items():
        actor2, critic2 = copy.deepcopy(actor1), copy.deepcopy(critic1)
        upd1 = FusedPPO2Update(actor1, critic1, 0.45, np.zeros(A), np.full(A, 5.0), "relu", max_grad_norm=max_norm)
        upd2 = FusedPPO2Update(actor2, critic2, 0.45, np.zeros(A), np.full(A, 5.0), "relu", max_grad_norm=max_norm)
        upd2.learn(s, a, a_lp, adv, vt, k_epochs=2, mini_batch=400, perm_key=1000)
        for e in range(2):
            for first in range(0, B, 400):
                upd1.grad_step(s, a, a_lp, adv, vt, first, min(400, B - first), perm_key=1000 + e)
                upd1.adam_step()
        assert upd2.step_count == upd1.step_count == 10
        assert torch.equal(upd1.params.flat, upd2.params.flat), max_norm


@pytest.mark.gpu
def test_wide_nets_are_rejected_loudly():
    from reinforcementlearningplatform_b200 import _lib
    from reinforcementlearningplatform_b200.learn import FusedPPO2Update, fused_supported
    from reinforcementlearningplatform_b200.ppo2 import dppo2_nets
    actor, critic = dppo2_nets(41, 2, np.array([-3.0, -1.0]), np.array([3.0, 2.0]), "cuda", hidden=256)
    assert not fused_supported(actor, critic)
    with pytest.raises(_lib.B200EnvError):
        FusedPPO2Update(actor, critic, actor.std, [-3.0, -1.0], [3.0, 2.0], "tanh_range")
