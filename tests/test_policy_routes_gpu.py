"""K-POLICY (csrc/policy.cu, policy_umma.cu, policy_umma16.cu) against a float64 restatement of choose_action, on every
kernel route.

Routes.  ``b200_policy_forward_packed`` ("umma") sends a net pair to ``policy_umma16.cu`` when ``policy_umma16_fits``
holds, else to one of the modes ``build_plan`` of ``policy_umma.cu`` picks: weights resident with the activations in
TMEM ("tmem"), resident with the activations in shared memory and one tile in flight ("smem1"; two tiles, ``cand == 1``,
is unreachable), or weights streamed through a TMA ring ("streamed").  ``_h_plan`` / ``_u_plan`` restate both host
plans line for line; ``test_route_restatement_matches_the_library`` holds them to ``b200_policy_workspace_bytes`` and
``test_rows_reach_every_route_and_branch`` (CPU) fails if ``ROWS`` stops reaching the branches listed there.  The fp32
FMA kernel ("fp32", ``policy.cu``) runs every row it holds (layers <= 64 wide, scalar std).

Bound.  Every output entry within ``C * 2^-24 * scale`` of float64, C = ``C_FP32`` or ``C_UMMA``.  ``_net64`` computes
the scale of a net's output in units of 2^-24 by a float64 forward pass alongside the real one:
  * layer l adds ``|W_l| |h_{l-1}| + |b_l|`` (the condition of its sum) to the input's error carried through ``|W_l|``;
  * each hidden activation adds ``TANH_UNITS``: the SFU tanh (<= 4e-7, about 7 units) and the rounding of the fp16 or
    TF32 operand pair the next layer multiplies (|x| <= 1, <= 6e-8); tanh itself is 1-Lipschitz;
  * every layer multiplied as fp16 hi / lo pairs (each layer after a net's first, on policy_umma16.cu and in the
    streamed mode) adds ``2^-14 max|W_l| sum_k |h_{l-1,k}|``.  ``policy_pack16_kernel`` / ``policy_pack_kernel`` scale
    the whole layer by one power of two that puts max|W_l| just below 2^14, so the lo half of a small weight stops at
    fp16's subnormal spacing 2^-24 of that scale: its error is relative to the layer's largest weight, not to its own
    row (2^-24 * 2^-14 max|W_l| per weight);
  * the tanh_range head multiplies by the gain and adds the SFU term; the action adds the rounding of
    ``mean + std eps``; the log-prob carries ``|a - mean| / std^2`` times the error of ``a - mean`` plus its own
    rounding.
An all-zero head must return its bias bit for bit.  The exploration draw is restated exactly (``philox4x32_10``,
``policy_noise``) and pinned to the Random123 known answers and to the C oracle."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

EPS32 = 2.0 ** -24
# 10x the largest ratio |out - out64| / (2^-24 scale) measured over the sweep below on a B200 (1000 W power limit):
# 6.68 for policy.cu (the value of the 33-64-1 critic), 6.24 for the tcgen05 kernels (the value of the one-layer 1-1
# critic, policy_umma16.cu)
C_FP32 = 67.0
C_UMMA = 63.0
TANH_UNITS = 8.0
# |z - z64| of the in-kernel Box-Muller draw (lg2 / sqrt / sin / cos .approx) against float64 on the same uniforms:
# 10x the 1.19e-5 measured on the same B200 (every route alike)
BM_BOUND = 1.2e-4

# actor dims, critic dims, actor head, per-dimension std; the route each row takes is in the comment and is asserted by
# test_rows_reach_every_route_and_branch
ROWS = {
    "ref": ((6, 64, 64, 32, 8), (6, 64, 32, 1), "relu", False),                      # umma16: the recorded nets
    "k2_deep_critic": ((9, 16, 3), (9, 16, 16, 16, 1), "identity", False),          # umma16: 2 k-steps, N = 16
    "k3_w48": ((20, 48, 48, 5), (20, 48, 1), "tanh_range", True),                   # umma16: 3 k-steps, N = 48
    "k4_eight_layers": ((32, 64, 64, 64, 16), (32, 64, 64, 64, 1), "relu", True),  # umma16: 4 k-steps, 8 layers
    "s1_w17": ((1, 17, 1), (1, 1), "identity", False),                              # umma16: N = 32 from 17
    "one_layer_actor": ((4, 2), None, "relu", False),                               # umma16
    "s33": ((33, 64, 4), (33, 64, 1), "tanh_range", False),                         # tmem
    "s41": ((41, 64, 64, 32, 8), (41, 64, 32, 1), "relu", False),                   # tmem
    "w80": ((6, 80, 80, 4), (6, 80, 1), "identity", True),                          # smem1: tail chunk
    "w65": ((16, 65, 2), (16, 65, 1), "relu", False),                               # smem1: tail chunk
    "s100": ((100, 64, 3), None, "tanh_range", False),                              # smem1: 4 input chunks
    "dppo2": ((41, 256, 256, 2), (41, 256, 256, 1), "tanh_range", True),            # streamed: the DPPO2 demo nets
    "w144_200": ((7, 144, 200, 10), (7, 144, 200, 1), "relu", False),              # streamed: tail chunks, A = 10
    "s256": ((256, 256, 16), (256, 256, 1), "identity", True),                      # streamed: 8 input chunks
}
HEADS = ("identity", "relu", "tanh_range")
WEIGHTS = ("default", "head_small", "x4", "row_tiny", "zero_head")
OBS = ("uniform", "mixed", "zeros")
N_SMALL = (1, 127, 128, 129, 4 * 128 + 1)
N_LARGE = 148 * 4 * 128 * 2 + 77       # several groups of the persistent loop in every CTA of both tcgen05 kernels


def _fp32_holds(row):
    actor, critic, _, std_vec = ROWS[row]
    return not std_vec and all(o <= 64 for dims in (actor, critic) if dims for o in dims[1:])


# ------------------------------------------------------------------------------------------------ host plans (CPU)
def _h_plan(actor, critic):
    """policy_umma16.cu:380-423 (h_add_net, h_build_plan): the per-layer (K, N, first, role) list, image bytes and bias
    floats, or None where it returns B200ENV_ESIZE (policy_umma16_fits false)"""
    layers, img, bias = [], 0, 0
    for dims, is_actor in ((actor, True), (critic, False)):
        if dims is None:
            continue
        if not 1 <= len(dims) - 1 <= 4:                                    # :381
            return None
        for l in range(len(dims) - 1):
            if len(layers) >= 8:                                           # :383 H_MAX_LAYERS
                return None
            i, o, last = dims[l], dims[l + 1], l + 2 == len(dims)
            if i < 1 or o < 1 or o > 64 or (l == 0 and i > 32) or (last and o > 16):   # :387
                return None
            K = (i + 7) // 8 * 8 if l == 0 else layers[-1]["N"]           # :389
            N = (o + 15) // 16 * 16                                        # :390
            layers.append(dict(K=K, N=N, first=l == 0, role=(1 if is_actor else 2) if last else 0, f16=l > 0))
            img += K * N * (8 if l == 0 else 4)                            # :396
            bias += N                                                      # :398
    bias += 8                                                              # :414 zs
    smem = 128 + (img + 127) // 128 * 128 + (bias * 4 + 127) // 128 * 128 + 4 * 16 * 128 * 4 + 512   # :415-421
    if smem > 227 * 1024:                                                  # :422
        return None
    return dict(mode="umma16", layers=layers, ws=(img + 127) // 128 * 128 + bias * 4)          # :435


def _u_plan(actor, critic):
    """policy_umma.cu:616-695 (add_net, build_plan): cand 0 -> "tmem", 1 -> "smem2", 2 -> "smem1", 3 -> "streamed";
    None where it returns B200ENV_ESIZE"""
    layers, img, bias = [], 0, 0
    for dims, is_actor in ((actor, True), (critic, False)):
        if dims is None:
            continue
        if not 1 <= len(dims) - 1 <= 4:                                    # :617
            return None
        for l in range(len(dims) - 1):
            if len(layers) >= 8:                                           # :619
                return None
            i, o, last = dims[l], dims[l + 1], l + 2 == len(dims)
            if i < 1 or o < 1 or i > 256 or o > 256 or (last and o > 16):  # :621, :624
                return None
            K = (i + 7) // 8 * 8 if l == 0 else layers[-1]["N"]           # :626
            N = (o + 15) // 16 * 16                                        # :627
            layers.append(dict(K=K, N=N, first=l == 0, role=(1 if is_actor else 2) if last else 0, f16=False))
            img += K * N * 8                                               # :632
            bias += N                                                      # :634
    bias += 8                                                              # :651
    nmax = max([16] + [L["N"] for L in layers])                            # :652-656
    kmax = max([8] + [L["K"] for L in layers])
    bias_bytes = (bias * 4 + 127) // 128 * 128                             # :657
    chunks = (kmax + 31) // 32                                             # :658
    scr = 2 * 16 * 128 * 4 + 512                                           # :661
    for cand in range(4):                                                  # :662
        slots, streamed, a_tmem = (2 if cand <= 1 else 1), cand == 3, cand == 0
        nbuf_log2 = 2 if streamed else (2 if chunks > 2 else 1)            # :664
        if a_tmem and chunks > (1 << nbuf_log2):                           # :665
            continue
        a_bytes = 0 if a_tmem else slots * (1 << nbuf_log2) * 32768        # :666
        b_bytes = 4 * nmax * 64 if streamed else (img + 127) // 128 * 128  # :667-668
        total = 256 + a_bytes + b_bytes + bias_bytes + scr                 # :669
        cols = slots * (2 * nmax + (2 * 32 * (1 << nbuf_log2) if a_tmem else 0))   # :670-671
        pow2 = 32
        while pow2 < cols:                                                 # :672
            pow2 *= 2
        if total > 227 * 1024 or pow2 > 512:                               # :673
            continue
        if streamed:                                                       # :674-685
            for L in layers:
                L["f16"] = not L["first"]
            img = sum(L["K"] * L["N"] * (4 if L["f16"] else 8) for L in layers)
        mode = ("tmem", "smem2", "smem1", "streamed")[cand]
        return dict(mode=mode, layers=layers, ws=(img + 127) // 128 * 128 + bias * 4)   # policy_umma.cu:703
    return None


def route(actor, critic):
    """the plan of b200_policy_forward_packed for this pair (policy_umma.cu:728: policy_umma16_fits first)"""
    return _h_plan(actor, critic) or _u_plan(actor, critic)


def _launches():
    """(row, actor dims, critic dims) of every launch the GPU tests make: the joint pair and, where a row has both
    nets, the actor-only and critic-only launches"""
    out = []
    for name, (actor, critic, _, _) in ROWS.items():
        out.append((name, actor, critic))
        if actor and critic:
            out += [(name, actor, None), (name, None, critic)]
    return out


def _mlp(dims):
    """b200_mlp with the dims only: b200_policy_workspace_bytes reads no weights"""
    from reinforcementlearningplatform_b200 import _lib
    m = _lib.MLP()
    m.n_layers = len(dims) - 1
    for i, d in enumerate(dims):
        m.dims[i] = d
    return m


def test_route_restatement_matches_the_library():
    """The workspace size tells the resident modes (8 bytes per weight) from umma16 / streamed (4 bytes per weight after
    a net's first layer); the finer splits rest on the line-for-line restatement above."""
    from reinforcementlearningplatform_b200 import _lib
    lib = _lib.load()
    pairs = {(a, c) for _, a, c in _launches()}
    # and a grid across the boundaries of both plans, rejected nets included (both return 0)
    for s in (1, 8, 9, 32, 33, 64, 65, 256, 257):
        for w in (16, 17, 48, 64, 65, 112, 128, 200, 256, 257):
            for A in (1, 16, 17):
                pairs.add(((s, w, A), (s, w, 1)))
                pairs.add(((s, w, w, w, A), None))
    for actor, critic in sorted(pairs, key=str):
        ra = None if actor is None else C.byref(_mlp(actor))
        rc = None if critic is None else C.byref(_mlp(critic))
        plan = route(actor, critic)
        assert int(lib.b200_policy_workspace_bytes(ra, rc)) == (plan["ws"] if plan else 0), (actor, critic)


def test_rows_reach_every_route_and_branch():
    modes, k16, n16, depths, nlayers = set(), set(), set(), set(), set()
    tail, chunked, A_seen, blocks, heads, stds = set(), set(), set(), set(), set(), set()
    widths, fields, kinds = set(), set(), set()
    for name, actor, critic in _launches():
        plan = route(actor, critic)
        joint = route(ROWS[name][0], ROWS[name][1])
        # a split launch takes the joint launch's route, so the bit-equality of split and joint launches is meaningful
        assert plan["mode"] == joint["mode"], (name, actor, critic)
        modes.add(plan["mode"])
        kinds.add("joint" if actor and critic else "actor" if actor else "critic")
        nlayers.add(len(plan["layers"]))
        for dims in (actor, critic):
            if dims:
                depths.add((plan["mode"], len(dims) - 1))
                widths.update(dims[1:-1])
                fields.add(dims[0])
        for L in plan["layers"]:
            if plan["mode"] == "umma16":
                if L["first"]:
                    k16.add(L["K"] // 8)
                if L["role"] == 0:
                    n16.add(L["N"])
            elif plan["mode"] in ("smem1", "streamed"):
                if L["role"] == 0 and L["N"] % 32:
                    tail.add(plan["mode"])                                   # epi_tanh_chunk<8, false>
                if L["first"] and L["K"] > 32:
                    chunked.add(plan["mode"])
        if actor:
            A_seen.add(actor[-1])
            blocks.add(((actor[-1] + 3) // 4, actor[-1] % 4 != 0))
            heads.add(ROWS[name][2])
            stds.add(ROWS[name][3])
    assert modes == {"umma16", "tmem", "smem1", "streamed"}                  # never "smem2" (cand == 1)
    assert k16 == {1, 2, 3, 4} and n16 == {16, 32, 48, 64}
    assert {d for m, d in depths if m == "umma16"} == {1, 2, 3, 4} and max(nlayers) == 8
    assert tail == {"smem1", "streamed"} and chunked == {"smem1", "streamed"}
    assert {1, 3, 4, 5, 8, 16} <= A_seen
    assert {b for b, _ in blocks} == {1, 2, 3, 4} and (1, True) in blocks and (2, True) in blocks and (3, True) in blocks
    assert heads == set(HEADS) and stds == {False, True}
    assert kinds == {"joint", "actor", "critic"}
    assert any(c and a and len(c) > len(a) for a, c, _, _ in ROWS.values())  # a critic deeper than its actor
    assert {64, 65} <= widths and {32, 33} <= fields
    assert sum(_fp32_holds(r) for r in ROWS) >= 6
    # cand == 1 (two tiles with the activations in shared memory) is reached by no shape (DESIGN section 3): with at most
    # two input chunks cand 0 fits the TMEM columns and fails only on shared memory, which cand 1 needs more of; with
    # more, two rings of four 32 KB chunks exceed shared memory
    for s in (1, 8, 32, 33, 64, 65, 100, 128, 256):
        for d in (1, 2, 3, 4):
            for w in (8, 16, 17, 32, 48, 64, 65, 80, 96, 112, 113, 128, 144, 160, 192, 224, 256):
                for A in (1, 8, 16):
                    for crit in (None, 1):
                        a = (s,) + (w,) * (d - 1) + (A,)
                        c = None if crit is None else (s,) + (w,) * (d - 1) + (1,)
                        plan = route(a, c)
                        assert plan is None or plan["mode"] != "smem2", (a, c)


# ------------------------------------------------------------------------------------------------ Philox (CPU)
_M32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """Philox4x32-10 (Salmon et al., SC'11) over arrays: ctr [4, m], key [2, m] (uint32-valued) -> [4, m] uint64"""
    c = [np.asarray(x, np.uint64) & _M32 for x in ctr]
    k0, k1 = (np.asarray(x, np.uint64) & _M32 for x in key)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & _M32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & _M32]
        k0 = (k0 + np.uint64(0x9E3779B9)) & _M32
        k1 = (k1 + np.uint64(0xBB67AE85)) & _M32
    return np.stack(c)


def policy_noise(seed, step, idx, A):
    """policy_sample_store_fn (policy_common.cuh): the eps of dimensions 0..A-1 for global instance indices idx, in
    float64 from the same 32-bit words.  Key (seed_lo, seed_hi ^ B200_POLICY_KEY_DOMAIN), counter (idx_lo, idx_hi,
    step_lo, ((step >> 32) << 8) + g) for block g; word k of block g feeds dimension 4 g + k; Box-Muller on u1 =
    ((r0 >> 8) + 1) / 2^24 in (0, 1] and angle (r1 >> 8) 2 pi / 2^24 - pi."""
    idx = np.asarray(idx, np.uint64)
    m = idx.size
    key = [np.full(m, seed & 0xFFFFFFFF, np.uint64), np.full(m, (seed >> 32) ^ 0x504F4C49, np.uint64)]
    z = np.empty((A, m))
    for g in range((A + 3) // 4):
        c3 = ((((step >> 32) & 0xFFFFFFFF) << 8) + g) & 0xFFFFFFFF
        r = philox4x32_10([idx & _M32, idx >> np.uint64(32), np.full(m, step & 0xFFFFFFFF, np.uint64),
                           np.full(m, c3, np.uint64)], key)
        for h in range(2):
            u1 = ((r[2 * h] >> np.uint64(8)).astype(np.float64) + 1.0) / 2.0 ** 24
            ang = (r[2 * h + 1] >> np.uint64(8)).astype(np.float64) * (2 * math.pi / 2.0 ** 24) - math.pi
            rad = np.sqrt(-2.0 * np.log(u1))
            for q, v in ((2 * h, rad * np.cos(ang)), (2 * h + 1, rad * np.sin(ang))):
                if 4 * g + q < A:
                    z[4 * g + q] = v
    return z


def test_philox_known_answers_and_oracle(oracle_lib):
    from oracle import oracle
    kat = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
           ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
           ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
            (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]
    for ctr, key, want in kat:
        assert tuple(int(v) for v in philox4x32_10([[c] for c in ctr], [[k] for k in key])[:, 0]) == want
        assert tuple(int(v) for v in oracle.philox(ctr, key)) == want
    rng = np.random.default_rng(5)
    ctr, key = rng.integers(0, 2 ** 32, (4, 64), dtype=np.uint64), rng.integers(0, 2 ** 32, (2, 64), dtype=np.uint64)
    got = philox4x32_10(ctr, key)
    for j in range(64):
        assert np.array_equal(got[:, j], oracle.philox(ctr[:, j], key[:, j]).astype(np.uint64))


def test_policy_noise_restatement_is_standard_normal():
    z = policy_noise(7, 3, np.arange(1 << 16), 5)
    assert abs(z.mean()) < 0.01 and abs(z.std() - 1.0) < 0.01
    assert abs(np.corrcoef(z[0], z[1])[0, 1]) < 0.02 and abs(np.corrcoef(z[0], z[4])[0, 1]) < 0.02


# ------------------------------------------------------------------------------------------------ GPU helpers
def _nets(row, weights, seed):
    """(actor Linear list | None, critic Linear list | None) of the row with weight variant ``weights``"""
    actor, critic, _, _ = ROWS[row]
    torch.manual_seed(seed)
    out = []
    for dims in (actor, critic):
        if dims is None:
            out.append(None)
            continue
        lins = [torch.nn.Linear(i, o).cuda() for i, o in zip(dims[:-1], dims[1:])]
        with torch.no_grad():
            if weights == "head_small":            # the common PPO initialisation of the output layer
                lins[-1].weight.mul_(0.01)
                lins[-1].bias.mul_(0.01)
            elif weights == "x4":                  # saturates tanh
                for lin in lins:
                    lin.weight.mul_(4.0)
                    lin.bias.mul_(4.0)
            elif weights == "row_tiny":            # one output row 2^-20 of the rest, in an fp16-split layer where one exists
                lins[min(1, len(lins) - 1)].weight[0].mul_(2.0 ** -20)
            elif weights == "zero_head":
                lins[-1].weight.zero_()
        out.append(lins)
    return out


def _obs(kind, S, n, gen):
    u = torch.rand(S, n, device="cuda", generator=gen) * 2 - 1
    if kind == "mixed":                            # fields of scale 1e3 next to fields of scale 1e-3
        u = u * torch.where(torch.arange(S, device="cuda") % 2 == 0, 1e3, 1e-3)[:, None]
    elif kind == "zeros":                          # exact zeros of both signs
        u = torch.where(u < 0, -0.0, 0.0)
    return u.float().contiguous()


def _bounds(row):
    """a_min, a_max, std (float or per-dimension array) of the row"""
    actor, _, _, std_vec = ROWS[row]
    A = actor[-1] if actor else 1
    j = np.arange(A, dtype=np.float32)
    a_min, a_max = (-1.5 - 0.1 * j).astype(np.float32), (1.5 + 0.2 * j).astype(np.float32)
    std = np.linspace(0.3, 1.5, A).astype(np.float32) if std_vec else 0.7
    return a_min, a_max, std


def _policy(row, nets, precision, head=None, **kw):
    import reinforcementlearningplatform_b200 as rlp
    a_min, a_max, std = _bounds(row)
    return rlp.GaussianPolicy(nets[0], nets[1], a_min, a_max, std, precision=precision,
                              actor_out_act=head or ROWS[row][2], **kw)


def _net64(lins, x, f16):
    """float64 forward of the net's layers (head activation not applied) and the error scale of its output in units of
    2^-24 (module docstring).  x: [n, S] float64; f16: the layers after the first multiply fp16 pairs."""
    h, E = x, torch.zeros_like(x)
    for l, lin in enumerate(lins):
        W, b = lin.weight.detach().double(), lin.bias.detach().double()
        Wa, ha = W.abs(), h.abs()
        z = h @ W.T + b
        E = E @ Wa.T + ha @ Wa.T + b.abs()
        if f16 and l > 0:
            E = E + 2.0 ** -14 * float(Wa.max()) * ha.sum(1, keepdim=True)
        if l + 1 < len(lins):
            h, E = torch.tanh(z), E + TANH_UNITS
    return z, E


def _reference(row, nets, obs, eps, f16):
    """choose_action and the critic in float64 on the kernel's float32 inputs: dict of (value, scale) pairs"""
    actor, critic = nets
    _, _, head, _ = ROWS[row]
    a_min, a_max, std = _bounds(row)
    x = obs.double().T
    out = {}
    if actor:
        A = actor[-1].out_features
        z, Ez = _net64(actor, x, f16)
        lo = torch.as_tensor(a_min, dtype=torch.float64, device="cuda")
        hi = torch.as_tensor(a_max, dtype=torch.float64, device="cuda")
        sd = torch.as_tensor(np.broadcast_to(np.float32(std), (A,)).astype(np.float64), device="cuda")
        if head == "relu":
            mean, Em = torch.relu(z), Ez
        elif head == "identity":
            mean, Em = z, Ez
        else:
            off = (lo + hi) / 2
            mean = torch.tanh(z) * (hi - off) + off
            Em = (hi - off) * (Ez + TANH_UNITS + 1) + off.abs() + mean.abs()
        e = eps.double().T
        act = torch.minimum(torch.maximum(mean + sd * e, lo), hi)
        Ea = Em + (sd * e).abs() + act.abs()
        d = act - mean
        lp = -d * d / (2 * sd * sd) - torch.log(sd) - 0.5 * math.log(2 * math.pi)
        El = d.abs() / (sd * sd) * (Ea + Em + d.abs()) + 4 * (d * d / (2 * sd * sd) + torch.log(sd).abs() + 1.0)
        out.update(mean=(mean, Em), action=(act, Ea), log_prob=(lp, El))
    if critic:
        z, Ez = _net64(critic, x, f16)
        out["value"] = (z[:, :1], Ez[:, :1])
    return out


def _ratios(got, ref):
    """max |got - ref| / (2^-24 scale) per output"""
    r = {}
    for k, (v, E) in ref.items():
        g = got[k].double()
        g = g.T if g.dim() == 2 else g[:, None]
        assert torch.isfinite(g).all(), k
        r[k] = float(((g - v).abs() / (EPS32 * E)).max())
    return r


# ------------------------------------------------------------------------------------------------ float64 (GPU)
def _cases():
    cases = [(w, o, N_SMALL[i % len(N_SMALL)]) for i, (w, o) in enumerate((w, o) for w in WEIGHTS for o in OBS)]
    cases += [("default", "uniform", n) for n in N_SMALL + (N_LARGE,)] + [("head_small", "uniform", N_LARGE)]
    return cases


ROUTE_CASES = [(r, "umma") for r in ROWS] + [(r, "fp32") for r in ROWS if _fp32_holds(r)]


@pytest.mark.gpu
@pytest.mark.parametrize("row,precision", ROUTE_CASES)
def test_matches_float64_choose_action(row, precision):
    plan = route(ROWS[row][0], ROWS[row][1])
    f16 = precision == "umma" and plan["mode"] in ("umma16", "streamed")
    bound = C_FP32 if precision == "fp32" else C_UMMA
    gen = torch.Generator(device="cuda").manual_seed(17)
    worst, bad, built = {}, [], {}
    for weights, obs_kind, n in _cases():
        if weights not in built:
            nets = _nets(row, weights, seed=len(built))
            built[weights] = (nets, _policy(row, nets, precision))
        nets, pol = built[weights]
        S = (nets[0] or nets[1])[0].in_features
        obs = _obs(obs_kind, S, n, gen)
        A = nets[0][-1].out_features
        eps = torch.randn(A, n, device="cuda", generator=gen)
        got = pol(obs, noise=eps, want_mean=True)
        torch.cuda.synchronize()
        ref = _reference(row, nets, obs, eps, f16)
        r = _ratios(got, ref)
        for k, v in r.items():
            worst[k] = max(worst.get(k, 0.0), v)
            if not v <= bound:
                bad.append((weights, obs_kind, n, k, round(v, 1)))
        if weights == "zero_head":                 # the head's bias, bit for bit
            if nets[0] and ROWS[row][2] != "tanh_range":
                b = nets[0][-1].bias.detach()
                b = torch.relu(b) if ROWS[row][2] == "relu" else b
                assert torch.equal(got["mean"], b[:, None].expand(A, n)), (row, precision)
            if nets[1]:
                assert torch.equal(got["value"], nets[1][-1].bias.detach().expand(n)), (row, precision)
    print(f"ratio {precision} {plan['mode'] if precision == 'umma' else 'fp32'} {row} "
          + " ".join(f"{k}={v:.3f}" for k, v in sorted(worst.items())))
    assert not bad, (row, precision, bound, bad)


# ------------------------------------------------------------------------------------------------ the draw (GPU)
SEEDS, OFFSETS, STEPS = (9, (1 << 32) + 0x1234567), (0, (1 << 32) - 150), (0, 1, (1 << 32) + 3)


@pytest.mark.gpu
@pytest.mark.parametrize("row,precision", ROUTE_CASES)
def test_exploration_draw_is_the_restated_philox_box_muller(row, precision):
    """noise=None: the kernel's eps = action / std (mean = 0 exactly: zero head, identity head, a clamp that never
    binds) equals the float64 Box-Muller of the restated Philox words within BM_BOUND, for seeds >= 2^32, steps 0, 1 and
    2^32 + 3 (set through GaussianPolicy.step), and instance offsets across 2^32"""
    import reinforcementlearningplatform_b200 as rlp
    actor, critic, _, std_vec = ROWS[row]
    nets = _nets(row, "zero_head", seed=3)
    with torch.no_grad():
        nets[0][-1].bias.zero_()
    A, n = actor[-1], 300
    std = np.linspace(0.3, 1.5, A).astype(np.float32) if std_vec else np.float32(0.7)
    sd = np.broadcast_to(std, (A,)).astype(np.float64)[:, None]
    obs = torch.rand(actor[0], n, device="cuda") * 2 - 1
    worst = 0.0
    for seed in SEEDS:
        for off in OFFSETS:
            pol = rlp.GaussianPolicy(nets[0], nets[1], np.full(A, -1e4, np.float32), np.full(A, 1e4, np.float32), std,
                                     precision=precision, actor_out_act="identity", seed=seed, env_index_offset=off)
            for step in STEPS:
                pol.step = step
                out = pol(obs, want_mean=True)
                assert pol.step == step + 1
                assert not out["mean"].any()
                z = out["action"].double().cpu().numpy() / sd
                z64 = policy_noise(seed, step, off + np.arange(n), A)
                err = float(np.abs(z - z64).max())
                worst = max(worst, err)
                assert err <= BM_BOUND, (row, precision, seed, off, step, err)
    print(f"box-muller {precision} {row} max|z - z64| = {worst:.3e}")


# ------------------------------------------------------------------------------------------------ isolation (GPU)
SENTINEL = 0x7FC0DEAD       # a NaN payload no kernel produces (their NaNs are the canonical 0x7FFFFFFF)


def _canary_buffers(A, n, critic, pad=256):
    """the outputs as views into larger buffers filled with SENTINEL; pad > one 128-instance tile"""
    bufs, views = {}, {}
    shapes = [(k, (A, n)) for k in ("action", "log_prob", "mean") if A] + ([("value", (n,))] if critic else [])
    for k, shape in shapes:
        size = int(np.prod(shape))
        big = torch.full((pad + size + pad,), SENTINEL, dtype=torch.int32, device="cuda")
        bufs[k] = (big, pad, size)
        views[k] = big[pad:pad + size].view(torch.float32).view(shape)
    return bufs, views


@pytest.mark.gpu
@pytest.mark.parametrize("row,precision", ROUTE_CASES)
def test_writes_stay_inside_the_outputs_and_rows_are_independent(row, precision):
    """Canaries around every output of a ragged launch; an instance's outputs do not depend on n, on its position in
    the batch or (sampled) on the shard; actor-only and critic-only launches give the joint launch's bits"""
    actor, critic, _, _ = ROWS[row]
    nets = _nets(row, "default", seed=1)
    pol = _policy(row, nets, precision, seed=4)
    S, A, n = (actor or critic)[0], actor[-1] if actor else 0, 513
    gen = torch.Generator(device="cuda").manual_seed(2)
    obs = _obs("uniform", S, n, gen)
    eps = torch.randn(A, n, device="cuda", generator=gen) if A else None
    for noise in (eps, None):
        bufs, views = _canary_buffers(A, n, critic)
        pol(obs, noise=noise, **views)
        torch.cuda.synchronize()
        for k in views:
            big, pad, size = bufs[k]
            assert bool((big[:pad] == SENTINEL).all()) and bool((big[pad + size:] == SENTINEL).all()), (row, k, "outside")
            assert not bool((big[pad:pad + size] == SENTINEL).any()), (row, k, "inside")
    full = pol(obs, noise=eps, want_mean=True)
    for a, b in ((0, 1), (127, 256), (300, 513)):
        part = pol(obs[:, a:b].contiguous(), noise=None if eps is None else eps[:, a:b].contiguous(), want_mean=True)
        for k, v in part.items():
            assert torch.equal(v, full[k][..., a:b]), (row, k, a, b)
    if actor:                                     # the sampled path: one shard at the matching env_index_offset
        pol.step = 7
        whole = pol(obs)["action"]
        shard = _policy(row, nets, precision, seed=4, env_index_offset=300)
        shard.step = 7
        assert torch.equal(shard(obs[:, 300:].contiguous())["action"], whole[:, 300:]), row
    if actor and critic:
        only_a = _policy(row, (nets[0], None), precision)(obs, noise=eps, want_mean=True)
        only_c = _policy(row, (None, nets[1]), precision)(obs)
        for k in ("action", "log_prob", "mean"):
            assert torch.equal(only_a[k], full[k]), (row, k)
        assert torch.equal(only_c["value"], full["value"]), row


# ------------------------------------------------------------------------------------------------ non-finite (GPU)
@pytest.mark.gpu
@pytest.mark.parametrize("row,precision", ROUTE_CASES)
def test_nan_observation_gives_nan_outputs_for_that_instance_only(row, precision):
    """torch's choose_action: a NaN in any observation field makes that instance's mean, action, log_prob and value NaN;
    every other instance keeps its bits.  +-Inf: only the isolation half (torch returns finite outputs there; the
    tensor-core routes split an infinite observation into hi = inf, lo = inf - inf = NaN)."""
    actor, critic, _, _ = ROWS[row]
    nets = _nets(row, "default", seed=5)
    pol = _policy(row, nets, precision)
    S, A, n = (actor or critic)[0], actor[-1] if actor else 0, 300
    gen = torch.Generator(device="cuda").manual_seed(6)
    obs = _obs("uniform", S, n, gen)
    eps = torch.randn(A, n, device="cuda", generator=gen) if A else None
    clean = pol(obs, noise=eps, want_mean=True)
    for bad, insts in ((float("nan"), (0, 5, 129, 299)), (float("inf"), (7, 130)), (float("-inf"), (8, 200))):
        dirty = obs.clone()
        for i in insts:
            dirty[(3 * i) % S, i] = bad
        got = pol(dirty, noise=eps, want_mean=True)
        keep = torch.ones(n, dtype=torch.bool, device="cuda")
        keep[list(insts)] = False
        for k, v in got.items():
            assert torch.equal(v[..., keep], clean[k][..., keep]), (row, precision, bad, k)
            if math.isnan(bad):
                assert bool(v[..., ~keep].isnan().all()), (row, precision, k)
        if not math.isnan(bad):
            print(f"{bad} observation {precision} {row}: "
                  + " ".join(f"{k} finite={bool(v[..., ~keep].isfinite().all())}" for k, v in sorted(got.items())))
