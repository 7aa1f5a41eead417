"""b200_policy_pack against a numpy restatement of the packed workspace, bit for bit, on every tcgen05 route.

For each launch of ``test_policy_routes_gpu.py`` (umma16, and policy_umma.cu's TMEM, smem1 and streamed modes) the whole
workspace is compared: the weight image, its padding to 128 bytes, the bias floats and the per-layer accumulator scales
(``zs``).  The workspace is filled with a sentinel byte first; bytes the packer does not own must keep it.

Layout (the comment of ``policy_pack_kernel``, policy_umma.cu):
  * 3xTF32 layers (a net's first; every layer of the resident modes): per k-step of 8 a hi and a lo plane of N * 32 bytes,
    element (n, k) at (k % 8 / 4) * N * 16 + n * 16 + (k % 4) * 4; hi = (bits + 0x1000) & 0xffffe000, lo = x - hi;
  * fp16-split layers (the others): the layer times 2^s with s = 14 - e, m = f 2^e (frexp) the layer's max |w|, s in
    [-100, 100] (s = 0 for an all-zero layer); per k-step of 16 a hi and a lo plane, element (n, k) at
    (k % 16 / 8) * N * 16 + n * 16 + (k % 8) * 2, hi = fp16(x), lo = fp16(x - hi), round to nearest;
  * the bias of a tanh layer times float32(2 log2 e); zs[l] = 2^-s, times 2 log2 e for tanh layers."""
import ctypes as C

import numpy as np
import pytest
import torch

from test_policy_routes_gpu import ROWS, _launches, _mlp, route

TWO_LOG2E = np.float32(2.885390081777927)
SENTINEL = 0xA5
# weight variants: torch's default initialisation; every layer so small / so large that s is clamped to +100 / -100; every
# weight zero (s = 0); one output row 2^-20 of the rest (its lo halves reach fp16's subnormals)
VARIANTS = ("default", "tiny", "huge", "zero", "row_tiny")
# actor and critic with different input widths: b200_policy_forward_packed rejects such a pair, but b200_policy_pack packs
# it, each first layer with its own in-features (the critic's narrower or wider than the actor's), on both routes
MISMATCHED = {
    "s8_critic_s6": ((8, 64, 2), (6, 64, 1)),                        # umma16
    "s6_critic_s8": ((6, 64, 2), (8, 64, 1)),                        # umma16
    "s41_critic_s33": ((41, 256, 256, 2), (33, 256, 256, 1)),        # streamed
}


def _pairs(row):
    """(actor dims, critic dims) of every launch of the row"""
    if row in MISMATCHED:
        return [MISMATCHED[row]]
    return [(a, c) for name, a, c in _launches() if name == row]


def _layers(dims, variant, gen):
    """[(W float32 [out, in], b float32 [out])] of a net"""
    out = []
    for i, o in zip(dims[:-1], dims[1:]):
        bound = 1.0 / np.sqrt(i)
        W = gen.uniform(-bound, bound, (o, i)).astype(np.float32)
        b = gen.uniform(-bound, bound, o).astype(np.float32)
        if variant in ("tiny", "huge"):        # max |W| = 0.75 2^-+115: s = 129 / -101 before the clamp
            W = (W * (0.75 * 2.0 ** (115 if variant == "huge" else -115) / np.abs(W).max())).astype(np.float32)
        elif variant == "zero":
            W[:] = 0.0
        elif variant == "row_tiny":
            W[0] *= np.float32(2.0 ** -20)
        out.append((W, b))
    return out


def _tf32_hi(x):
    return ((x.view(np.uint32).astype(np.uint64) + 0x1000) & 0xFFFFE000).astype(np.uint32)


def _scale_exp(W):
    m = float(np.abs(W).max()) if W.size else 0.0
    e = int(np.frexp(np.float32(m))[1]) if 0.0 < m < 3.0e38 else 14
    return min(100, max(-100, 14 - e))


def _restate(plan, nets):
    """the expected workspace bytes (uint8) of the plan for [(W, b)] of every layer in launch order"""
    layers = plan["layers"]
    ws = np.full(plan["ws"], SENTINEL, np.uint8)
    img = sum(L["K"] * L["N"] * (4 if L["f16"] else 8) for L in layers)
    bias = ws[(img + 127) // 128 * 128:].view(np.float32)
    w_off, b_off, zs_off = 0, 0, sum(L["N"] for L in layers)
    for li, (L, (W, b)) in enumerate(zip(layers, nets)):
        K, N = L["K"], L["N"]
        Wp = np.zeros((N, K), np.float32)
        Wp[:W.shape[0], :W.shape[1]] = W
        k, n = np.meshgrid(np.arange(K), np.arange(N), indexing="ij")
        w = Wp[n, k]
        if L["f16"]:
            s = _scale_exp(W)
            ws_ = w * np.float32(2.0 ** s)
            hi = ws_.astype(np.float16)
            lo = (ws_ - hi.astype(np.float32)).astype(np.float16)
            at = w_off + (k // 16) * N * 64 + (k % 16 // 8) * N * 16 + n * 16 + (k % 8) * 2
            for plane, v in ((0, hi), (N * 32, lo)):
                b2 = v.view(np.uint16)
                ws[at + plane] = (b2 & 0xFF).astype(np.uint8)
                ws[at + plane + 1] = (b2 >> 8).astype(np.uint8)
            w_off += K * N * 4
        else:
            s = 0
            hi = _tf32_hi(w)
            lo = w - hi.view(np.float32)
            at = w_off + (k // 8) * N * 64 + (k % 8 // 4) * N * 16 + n * 16 + (k % 4) * 4
            for plane, v in ((0, hi), (N * 32, lo.view(np.uint32))):
                for byte in range(4):
                    ws[at + plane + byte] = ((v >> (8 * byte)) & 0xFF).astype(np.uint8)
            w_off += K * N * 8
        bp = np.zeros(N, np.float32)
        bp[:b.size] = b
        tanh = L["role"] == 0
        bias[b_off:b_off + N] = bp * TWO_LOG2E if tanh else bp
        bias[zs_off + li] = (TWO_LOG2E if tanh else np.float32(1.0)) * np.float32(2.0 ** -s)
        b_off += N
    return ws


def _pack(actor, critic, nets):
    """b200_policy_pack of the launch into a sentinel-filled workspace of b200_policy_workspace_bytes"""
    from reinforcementlearningplatform_b200 import _lib
    lib = _lib.load()
    dev = [(torch.from_numpy(W).cuda(), torch.from_numpy(b).cuda()) for W, b in nets]
    mlps, at = [], 0
    for dims in (actor, critic):
        if dims is None:
            mlps.append(None)
            continue
        m = _lib.MLP()
        m.n_layers = len(dims) - 1
        for i, d in enumerate(dims):
            m.dims[i] = d
        for l in range(m.n_layers):
            m.w[l], m.b[l] = dev[at + l][0].data_ptr(), dev[at + l][1].data_ptr()
        at += m.n_layers
        mlps.append(m)
    refs = [None if m is None else C.byref(m) for m in mlps]
    need = int(lib.b200_policy_workspace_bytes(*refs))
    ws = torch.full((need,), SENTINEL, dtype=torch.uint8, device="cuda")
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(lib.b200_policy_pack(*refs, C.c_void_p(ws.data_ptr()), need, stream), "b200_policy_pack")
    torch.cuda.synchronize()
    return ws.cpu().numpy()


def test_mismatched_input_widths_keep_their_workspace_size():
    """the pairs above are routed and sized like any other (b200_policy_workspace_bytes is not 0 for them)"""
    from reinforcementlearningplatform_b200 import _lib
    lib = _lib.load()
    modes = set()
    for actor, critic in MISMATCHED.values():
        plan = route(actor, critic)
        modes.add(plan["mode"])
        assert int(lib.b200_policy_workspace_bytes(C.byref(_mlp(actor)), C.byref(_mlp(critic)))) == plan["ws"] > 0
    assert modes == {"umma16", "streamed"}


@pytest.mark.gpu
@pytest.mark.parametrize("row", list(ROWS) + list(MISMATCHED))
def test_packed_workspace_is_the_restated_layout(row):
    modes = set()
    keys = list(ROWS) + list(MISMATCHED)
    for variant in VARIANTS:
        gen = np.random.default_rng([keys.index(row), VARIANTS.index(variant)])
        for actor, critic in _pairs(row):
            plan = route(actor, critic)
            modes.add(plan["mode"])
            nets = (_layers(actor, variant, gen) if actor else []) + (_layers(critic, variant, gen) if critic else [])
            got = _pack(actor, critic, nets)
            want = _restate(plan, nets)
            assert got.size == want.size, (row, actor, critic)
            bad = np.flatnonzero(got != want)
            assert bad.size == 0, (row, variant, actor, critic, plan["mode"], bad[:8], got[bad[:8]], want[bad[:8]])
    print(f"pack {row} {sorted(modes)}: workspace bit-identical over {len(VARIANTS)} weight variants")
