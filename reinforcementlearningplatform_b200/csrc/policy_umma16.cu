// policy_umma16.cu -- K-POLICY for the reference's small nets with FOUR tiles in flight per SM.
//
// Same contract as policy_umma.cu (Proximal_Policy_Optimization2.choose_action, algorithm/policy_base/
// Proximal_Policy_Optimization2.py:69-76, critic forward :88-90; nets of utils/classes.py:529-615).  What the event trace
// of policy_umma.cu showed (profiles/r2/policy_umma.md): with the activations in TMEM as two TF32 planes a tile slot needs
// 256 tensor-memory columns (D ping, D pong, A hi, A lo), so only TWO 128-instance tiles fit in the 512 columns; each
// tile walks its seven layers as a strictly serial chain (MMA -> commit -> tcgen05.ld -> tanh -> tcgen05.st -> MMA ...,
// ~3500 cycles per layer) and with two chains in flight the tensor pipe idles 60 % and the epilogue warps half of the
// time: 0.33 ms per 1 M instances although neither the MMA issue rate (~0.08 ms) nor the epilogue's instruction count
// (~0.10 ms) asks for more than a third of that.
//
// This kernel halves a slot's footprint so that four chains overlap:
//   * hidden-layer operands are split into two FP16 halves instead of two TF32 halves: x = hi + lo with hi = fp16(x),
//     lo = fp16(x - hi): 22 significand bits, the same as the TF32 pair.  Activations are tanh outputs (|x| <= 1, absolute
//     error of the pair <= 6e-8); each layer's weights are pre-scaled by a power of two so that max |w| sits just below
//     2^14 (no fp16 overflow, no subnormal halves) and the accumulator is scaled back inside the epilogue's FFMA.  D still
//     accumulates A_lo W_hi + A_hi W_lo + A_hi W_hi in fp32 (tests: <= 5e-6 absolute, as before);
//   * 16-bit A operands pack two K elements per TMEM column: hi and lo planes of a 64-wide layer input take 32 + 32
//     columns, D 64 -> 128 columns per slot, four slots;
//   * kind::f16 MMAs cover K = 16 per instruction: half the tcgen05.mma count of kind::tf32;
//   * the first layer of each net multiplies the raw observations (any magnitude): it keeps the 3xTF32 form (one k-step).
// Warp roles (640 threads): warps 0-15 epilogue, four per slot (warp % 4 = the TMEM lane quadrant it may touch, thread =
// row); warps 16-19 issue the MMAs of slot 0-3 from one elected lane each; the whole weight image (44 KB for the
// 6-64-64-32-8 + 6-64-32-1 nets) is fetched once per CTA by a bulk copy.  Per slot and layer two mbarriers alternate:
// a_full (128 arrivals: the layer's input is in TMEM and the previous accumulator has been read) and d_ready
// (tcgen05.commit).
// Nets this kernel does not hold (a layer wider than 64, more than 32 observation fields) take policy_umma.cu.
#include <cuda_fp16.h>
#include "policy_common.cuh"
#include "umma_ptx.cuh"

namespace {
using namespace umma;

constexpr int H_THREADS = 640;
constexpr int H_SLOTS = 4, H_EPI_WARPS = 16;
constexpr int H_TILE = 128;
constexpr int H_MAX_LAYERS = 8;
constexpr uint32_t H_SLOT_COLS = 128, H_A_COL = 64, H_A_LO = 32;
constexpr float H_TWO_LOG2E = 2.885390081777927f;
constexpr uint32_t H_SMEM_LIMIT = 227 * 1024;

struct HLayer {
    int K, N;        // padded: first layer K to a multiple of 8 (TF32), others K = previous N; N to a multiple of 16
    int n_real, k_real;
    int role;        // 0 hidden (tanh), 1 actor output, 2 critic output
    int first;       // input = observations (3xTF32); else fp16-split
    int out_act;
    uint32_t w_off;  // byte offset of the layer's image; k-step kk at w_off + kk * N * 64 (hi plane N * 32 B, then lo)
    int b_off;
};

struct HPlan {
    int n_layers, S, A;
    uint32_t img_bytes;
    int bias_floats, zs_off;   // zs_off: per-layer accumulator scale (x 2 log2 e for tanh layers) inside the bias array
    uint32_t off_b, off_bias, off_scr, smem_bytes;
    HLayer L[H_MAX_LAYERS];
};

struct HArgs {
    HPlan p;
    PolicyIO io;
    const unsigned char *image;
    const float *bias;
};

struct HBar {
    static constexpr uint32_t a_full = 0;     // [4]
    static constexpr uint32_t d_ready = 32;   // [4]
    static constexpr uint32_t w_ready = 64;
    static constexpr uint32_t tmem_slot = 72;
    static constexpr uint32_t bytes = 128;
};

// 16 accumulator values of row r (already in registers) -> tanh -> fp16 hi / lo pairs -> the next layer's A operand
// (8 + 8 TMEM columns)
__device__ __forceinline__ void epi16_compute(const uint32_t (&v)[16], const float *bias_scaled, float zs, uint32_t a_hi_addr,
                                              uint32_t a_lo_addr) {
    float t[16];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const float4 b = *reinterpret_cast<const float4 *>(bias_scaled + 4 * q);
        t[4 * q + 0] = b.x; t[4 * q + 1] = b.y; t[4 * q + 2] = b.z; t[4 * q + 3] = b.w;
    }
    // tanh(x) = 1 - 2 / (2^t + 1), t = 2 log2(e) x; zs = 2 log2(e) / (the layer's weight scale)
#pragma unroll
    for (int j = 0; j < 16; ++j) t[j] = fmaf(__uint_as_float(v[j]), zs, t[j]);
    // one reciprocal for two activations: 1 / a = b / (a b), 1 / b = a / (a b); the exponent is clamped so that a b stays
    // finite (2^60 + 1: tanh is 1 to the last bit long before).  1.5 instead of 2 MUFU per activation, +2 issue slots:
    // 0.2218 vs 0.2255 ms per 1 M instances for one reciprocal each (A/B on one box, twice).
#pragma unroll
    for (int j = 0; j < 16; ++j) t[j] = fminf(t[j], 60.0f);
#pragma unroll
    for (int j = 0; j < 16; ++j) asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t[j]) : "f"(t[j]));
#pragma unroll
    for (int j = 0; j < 16; j += 2) {
        const float a = t[j] + 1.0f, b = t[j + 1] + 1.0f;
        float r;
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a * b));
        t[j] = r * b;
        t[j + 1] = r * a;
    }
#pragma unroll
    for (int j = 0; j < 16; ++j) t[j] = fmaf(-2.0f, t[j], 1.0f);
    uint32_t hi[8], lo[8];
#pragma unroll
    for (int p = 0; p < 8; ++p) {
        const __half2 h = __floats2half2_rn(t[2 * p], t[2 * p + 1]);          // .x (low half) = even k
        const float2 f = __half22float2(h);
        const __half2 l = __floats2half2_rn(t[2 * p] - f.x, t[2 * p + 1] - f.y);
        hi[p] = *reinterpret_cast<const uint32_t *>(&h);
        lo[p] = *reinterpret_cast<const uint32_t *>(&l);
    }
    tmem_st8(a_hi_addr, hi);
    tmem_st8(a_lo_addr, lo);
}

// hidden layer of NCH x 16 columns: the tcgen05.ld of chunk c + 1 is in flight while chunk c goes through the SFU
template <int NCH>
__device__ __forceinline__ void epi_hidden(uint32_t slot_t, const float *bias_scaled, float zs) {
    uint32_t v[2][16];
    tmem_ld<16>(slot_t, v[0]);
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
        tmem_wait_ld();
        if (c + 1 < NCH) tmem_ld<16>(slot_t + 16 * (c + 1), v[(c + 1) & 1]);
        epi16_compute(v[c & 1], bias_scaled + 16 * c, zs, slot_t + H_A_COL + 8 * c, slot_t + H_A_COL + H_A_LO + 8 * c);
    }
}

__global__ void __launch_bounds__(H_THREADS, 1)
policy_umma16_kernel(const __grid_constant__ HArgs a, int64_t n) {
    extern __shared__ __align__(128) unsigned char smem[];
    const HPlan &P = a.p;
    const uint32_t sbase = smem_u32(smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float *bias_s = reinterpret_cast<float *>(smem + P.off_bias);
    float *scr_all = reinterpret_cast<float *>(smem + P.off_scr);
    const float *dimc = scr_all + H_SLOTS * 16 * H_TILE;

    if (threadIdx.x == 0) {
        for (int s = 0; s < H_SLOTS; ++s) {
            mbar_init(sbase + HBar::a_full + s * 8, H_TILE);
            mbar_init(sbase + HBar::d_ready + s * 8, 1);
        }
        mbar_init(sbase + HBar::w_ready, 1);
        fence_barrier_init();
    }
    if (warp == H_EPI_WARPS) tmem_alloc(sbase + HBar::tmem_slot, 512);
    for (int j = threadIdx.x; j < P.bias_floats; j += H_THREADS) bias_s[j] = __ldg(a.bias + j);
    if (a.io.action) policy_dims_fill(a.io, P.A, scr_all + H_SLOTS * 16 * H_TILE, threadIdx.x, H_THREADS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t *>(smem + HBar::tmem_slot);
    const int64_t tiles = (n + H_TILE - 1) / H_TILE;
    const int64_t groups = (tiles + H_SLOTS - 1) / H_SLOTS;

    if (warp < H_EPI_WARPS) {
        // ======================================================================== epilogue: four warps per slot
        const int s = warp >> 2;
        const int r = (warp & 3) * 32 + lane;                         // row of the tile = TMEM lane
        const uint32_t slot_t = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)s * H_SLOT_COLS;
        float *scr = scr_all + s * (16 * H_TILE) + r;                  // the row's means: scr[j * H_TILE]
        const uint32_t af = sbase + HBar::a_full + s * 8, dr = sbase + HBar::d_ready + s * 8;
        uint32_t layers_done = 0;
        // xn: the first tile's observation fields.  These loads are dead (x8 is reloaded for every tile below and the
        // compiler drops them), but they steer ptxas: without them the kernel has the same instructions in another order
        // and measured 0.9 % slower (0.2208 vs 0.2189 ms per 1 M instances, five alternated runs each, B200 at 1000 W).
        float xn[8];
        {
            const int64_t t0 = (int64_t)blockIdx.x * H_SLOTS + s, i0 = t0 * H_TILE + r;
            const bool l0 = t0 < tiles && i0 < n;
#pragma unroll
            for (int e = 0; e < 8; ++e) xn[e] = (l0 && e < P.S) ? __ldg(a.io.obs + (int64_t)e * n + i0) : 0.0f;
        }
        for (int64_t grp = blockIdx.x; grp < groups; grp += gridDim.x) {
            const int64_t tile = grp * H_SLOTS + s;
            if (tile >= tiles) break;
            const int64_t i = tile * H_TILE + r;
            const bool live = i < n;
            int pending_A = 0;
            // the row's first 8 observation fields: fetched once per tile (both nets start from them)
            float x8[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) x8[e] = xn[e];
#pragma unroll
            for (int e = 0; e < 8; ++e) x8[e] = (live && e < P.S) ? __ldg(a.io.obs + (int64_t)e * n + i) : 0.0f;
            for (int li = 0; li < P.n_layers; ++li) {
                const HLayer &L = P.L[li];
                if (L.first) {
                    // observations -> TF32 hi / lo planes of the A region (zero-padded to K)
                    for (int q = 0; q < L.K / 8; ++q) {
                        uint32_t hi[8], lo[8];
#pragma unroll
                        for (int e = 0; e < 8; ++e) {
                            const int k = 8 * q + e;
                            const float x = q == 0 ? x8[e] : ((live && k < P.S) ? __ldg(a.io.obs + (int64_t)k * n + i) : 0.0f);
                            hi[e] = tf32_hi(x);
                            lo[e] = __float_as_uint(x - __uint_as_float(hi[e]));
                        }
                        tmem_st8(slot_t + H_A_COL + 8 * q, hi);
                        tmem_st8(slot_t + H_A_COL + H_A_LO + 8 * q, lo);
                    }
                    tmem_wait_st();
                    tc_fence_before();
                    mbar_arrive(af);
                }
                // the actor's sampling, deferred to here: the next net's first layer is already with the tensor core
                if (pending_A) {
                    if (live) policy_sample_store(a.io, n, i, pending_A, scr, H_TILE, dimc);
                    pending_A = 0;
                }
                mbar_wait(dr, layers_done & 1);
                tc_fence_after();
                ++layers_done;
                const float zs = bias_s[P.zs_off + li];
                if (L.role == 0) {
                    switch (L.N >> 4) {
                    case 1: epi_hidden<1>(slot_t, bias_s + L.b_off, zs); break;
                    case 2: epi_hidden<2>(slot_t, bias_s + L.b_off, zs); break;
                    case 3: epi_hidden<3>(slot_t, bias_s + L.b_off, zs); break;
                    default: epi_hidden<4>(slot_t, bias_s + L.b_off, zs); break;
                    }
                    tmem_wait_st();
                    tc_fence_before();
                    mbar_arrive(af);
                } else if (L.role == 1) {
                    uint32_t v[16];
                    tmem_ld<16>(slot_t, v);
                    tmem_wait_ld();
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        float m = fmaf(__uint_as_float(v[j]), zs, bias_s[L.b_off + j]);
                        if (L.out_act == 1) m = fmaxf(m, 0.0f);
                        scr[j * H_TILE] = m;
                    }
                    pending_A = L.n_real;
                    tc_fence_before();
                } else {
                    uint32_t v[1];
                    tmem_ld<1>(slot_t, v);
                    tmem_wait_ld();
                    if (live) __stcs(a.io.value + i, fmaf(__uint_as_float(v[0]), zs, bias_s[L.b_off]));
                    tc_fence_before();
                }
            }
            if (pending_A && live) policy_sample_store(a.io, n, i, pending_A, scr, H_TILE, dimc);
        }
    } else {
        // ======================================================================== MMA issuers: one elected lane per slot
        const uint32_t s = (uint32_t)(warp - H_EPI_WARPS);
        if (elect_one_sync()) {
            const uint32_t wbar = sbase + HBar::w_ready;
            if (s == 0) {   // the weight image, once per CTA
                mbar_expect_tx(wbar, P.img_bytes);
                for (uint32_t o = 0; o < P.img_bytes; o += 32768u) {
                    const uint32_t bytes = min(32768u, P.img_bytes - o);
                    bulk_g2s(sbase + P.off_b + o, a.image + o, bytes, wbar);
                }
            }
            mbar_wait(wbar, 0);
            const uint32_t slot_t = tmem_base + s * H_SLOT_COLS;
            const uint32_t desc_hi = (128u >> 4) | (1u << 14);                    // SBO = 128 B, descriptor version 1
            const uint32_t b_base16 = ((sbase + P.off_b) & 0x3FFFFu) >> 4;
            const uint32_t af = sbase + HBar::a_full + s * 8, dr = sbase + HBar::d_ready + s * 8;
            uint32_t phase = 0;
            for (int64_t grp = blockIdx.x; grp < groups; grp += gridDim.x) {
                if (grp * H_SLOTS + (int64_t)s >= tiles) break;
                for (int li = 0; li < P.n_layers; ++li) {
                    const HLayer &L = P.L[li];
                    const uint32_t N = (uint32_t)L.N;
                    const uint32_t blo16 = N * 2, kstep16 = N * 4;                // N * 32 B and N * 64 B, >> 4
                    uint32_t b_hi = (b_base16 + (L.w_off >> 4)) | (N << 16);      // LBO = N * 16 B
                    uint32_t a_hi = slot_t + H_A_COL, acc = 0;
                    mbar_wait(af, phase & 1u);
                    ++phase;
                    tc_fence_after();
                    if (L.first) {
                        const uint32_t idesc = umma_idesc_tf32(H_TILE, L.N);
                        for (int j = 0; j < (L.K >> 3); ++j) {
                            umma_tf32_ts(slot_t, a_hi + H_A_LO, b_hi, desc_hi, idesc, acc);        // small terms first
                            umma_tf32_ts(slot_t, a_hi, b_hi + blo16, desc_hi, idesc, 1u);
                            umma_tf32_ts(slot_t, a_hi, b_hi, desc_hi, idesc, 1u);
                            acc = 1u; a_hi += 8; b_hi += kstep16;
                        }
                    } else {
                        const uint32_t idesc = umma_idesc_f16(H_TILE, L.N);
                        for (int j = 0; j < (L.K >> 4); ++j) {
                            umma_f16_ts(slot_t, a_hi + H_A_LO, b_hi, desc_hi, idesc, acc);
                            umma_f16_ts(slot_t, a_hi, b_hi + blo16, desc_hi, idesc, 1u);
                            umma_f16_ts(slot_t, a_hi, b_hi, desc_hi, idesc, 1u);
                            acc = 1u; a_hi += 8; b_hi += kstep16;
                        }
                    }
                    umma_commit(dr);
                }
            }
        }
        __syncwarp();
    }
    tc_fence_before();
    __syncthreads();
    if (warp == H_EPI_WARPS) tmem_dealloc(tmem_base, 512);
}

// ------------------------------------------------------------------------------------------------ weight packing
struct HPackArgs {
    int n_layers, zs_off;
    HLayer L[H_MAX_LAYERS];
    const float *w[H_MAX_LAYERS];
    const float *b[H_MAX_LAYERS];
    unsigned char *image;
    float *bias;
};

// nn.Linear weights [n_real][k_real] -> the operand image.  First layers: TF32 hi / lo planes, per k-step of 8: element
// (n, k) at (k % 8 / 4) * N * 16 + n * 16 + (k % 4) * 4.  Other layers: weights times 2^s (s chosen per layer so that
// max |w| 2^s lies in [2^13, 2^14)), fp16 hi / lo planes, per k-step of 16: element (n, k) at (k % 16 / 8) * N * 16 +
// n * 16 + (k % 8) * 2.  Bias vector: tanh layers times 2 log2 e; zs[l] = 2^-s (times 2 log2 e for tanh layers).
__global__ void __launch_bounds__(256) policy_pack16_kernel(const __grid_constant__ HPackArgs a) {
    __shared__ float s_max[8];
    __shared__ int s_exp;
    const int li = blockIdx.y;
    if (li >= a.n_layers) return;
    const HLayer &L = a.L[li];
    const int total = L.K * L.N, real = L.k_real * L.n_real;
    int sexp = 0;
    if (!L.first) {
        float m = 0.0f;
        for (int e = threadIdx.x; e < real; e += blockDim.x) m = fmaxf(m, fabsf(__ldg(a.w[li] + e)));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        if ((threadIdx.x & 31) == 0) s_max[threadIdx.x >> 5] = m;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < 8; ++w) m = fmaxf(m, s_max[w]);
            int e = 0;
            if (m > 0.0f && m < 3.0e38f) frexpf(m, &e);      // m = f 2^e, f in [0.5, 1)
            else e = 14;
            int sx = 14 - e;
            sx = sx > 100 ? 100 : (sx < -100 ? -100 : sx);
            s_exp = sx;
        }
        __syncthreads();
        sexp = s_exp;
    }
    const float scale = ldexpf(1.0f, sexp);
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
        const int k = e / L.N, nn = e - k * L.N;
        const float w = (nn < L.n_real && k < L.k_real) ? __ldg(a.w[li] + (int64_t)nn * L.k_real + k) : 0.0f;
        if (L.first) {
            const uint32_t hi = tf32_hi(w);
            unsigned char *ks = a.image + L.w_off + (uint32_t)(k / 8) * (uint32_t)L.N * 64;
            const uint32_t in_plane = (uint32_t)((k & 7) >> 2) * (uint32_t)L.N * 16 + (uint32_t)nn * 16 + (uint32_t)(k & 3) * 4;
            *reinterpret_cast<uint32_t *>(ks + in_plane) = hi;
            *reinterpret_cast<float *>(ks + (uint32_t)L.N * 32 + in_plane) = w - __uint_as_float(hi);
        } else {
            const float ws = w * scale;
            const __half hi = __float2half_rn(ws);
            const __half lo = __float2half_rn(ws - __half2float(hi));
            unsigned char *ks = a.image + L.w_off + (uint32_t)(k / 16) * (uint32_t)L.N * 64;
            const uint32_t in_plane = (uint32_t)((k & 15) >> 3) * (uint32_t)L.N * 16 + (uint32_t)nn * 16 + (uint32_t)(k & 7) * 2;
            *reinterpret_cast<__half *>(ks + in_plane) = hi;
            *reinterpret_cast<__half *>(ks + (uint32_t)L.N * 32 + in_plane) = lo;
        }
    }
    if (blockIdx.x == 0) {
        for (int j = threadIdx.x; j < L.N; j += blockDim.x) {
            const float b = j < L.n_real ? __ldg(a.b[li] + j) : 0.0f;
            a.bias[L.b_off + j] = L.role == 0 ? b * H_TWO_LOG2E : b;
        }
        if (threadIdx.x == 0) a.bias[a.zs_off + li] = (L.role == 0 ? H_TWO_LOG2E : 1.0f) * ldexpf(1.0f, -sexp);
    }
}

// ------------------------------------------------------------------------------------------------ host side
int h_add_net(const b200_mlp *m, bool is_actor, HPlan *P, const float **w, const float **b) {
    if (m->n_layers < 1 || m->n_layers > 4) return B200ENV_ESIZE;
    for (int l = 0; l < m->n_layers; ++l) {
        if (P->n_layers >= H_MAX_LAYERS) return B200ENV_ESIZE;
        const int in = m->dims[l], out = m->dims[l + 1];
        HLayer &L = P->L[P->n_layers];
        const bool last = l + 1 == m->n_layers;
        if (in < 1 || out < 1 || out > 64 || (l == 0 && in > 32) || (last && out > 16)) return B200ENV_ESIZE;
        L.first = l == 0;
        L.K = l == 0 ? (in + 7) / 8 * 8 : P->L[P->n_layers - 1].N;
        L.N = (out + 15) / 16 * 16;
        L.n_real = out;
        L.k_real = in;
        L.role = last ? (is_actor ? 1 : 2) : 0;
        L.out_act = m->out_act == 2 ? 0 : m->out_act;
        L.w_off = P->img_bytes;
        P->img_bytes += (uint32_t)L.K * (uint32_t)L.N * (l == 0 ? 8u : 4u);
        L.b_off = P->bias_floats;
        P->bias_floats += L.N;
        if (w) w[P->n_layers] = m->w[l];
        if (b) b[P->n_layers] = m->b[l];
        ++P->n_layers;
    }
    return B200ENV_OK;
}

int h_build_plan(const b200_mlp *actor, const b200_mlp *critic, HPlan *P, const float **w, const float **b) {
    *P = HPlan{};
    int rc;
    if (actor && (rc = h_add_net(actor, true, P, w, b))) return rc;
    if (critic && (rc = h_add_net(critic, false, P, w, b))) return rc;
    P->S = actor ? actor->dims[0] : critic->dims[0];
    P->A = actor ? actor->dims[actor->n_layers] : 0;
    P->zs_off = P->bias_floats;
    P->bias_floats += H_MAX_LAYERS;
    const uint32_t bias_bytes = ((uint32_t)P->bias_floats * 4 + 127) / 128 * 128;
    const uint32_t b_bytes = (P->img_bytes + 127) / 128 * 128;
    const uint32_t scr_bytes = H_SLOTS * 16 * H_TILE * 4 + 512;
    P->off_b = HBar::bytes;
    P->off_bias = P->off_b + b_bytes;
    P->off_scr = P->off_bias + bias_bytes;
    P->smem_bytes = P->off_scr + scr_bytes;
    return P->smem_bytes > H_SMEM_LIMIT ? B200ENV_ESIZE : B200ENV_OK;
}

} // namespace

bool policy_umma16_fits(const b200_mlp *actor, const b200_mlp *critic) {
    HPlan P;
    return h_build_plan(actor, critic, &P, nullptr, nullptr) == B200ENV_OK;
}

size_t policy_umma16_workspace_bytes(const b200_mlp *actor, const b200_mlp *critic) {
    HPlan P;
    if (h_build_plan(actor, critic, &P, nullptr, nullptr)) return 0;
    return (size_t)(P.img_bytes + 127) / 128 * 128 + (size_t)P.bias_floats * 4;
}

int policy_umma16_pack(const b200_mlp *actor, const b200_mlp *critic, void *workspace, size_t bytes, cudaStream_t stream) {
    HPackArgs pa = {};
    HPlan P;
    int rc = h_build_plan(actor, critic, &P, pa.w, pa.b);
    if (rc) return rc;
    for (int l = 0; l < P.n_layers; ++l)
        if (!pa.w[l] || !pa.b[l]) return B200ENV_ENULL;
    const size_t img = (size_t)(P.img_bytes + 127) / 128 * 128;
    if (!workspace) return B200ENV_ENULL;
    if (bytes < img + (size_t)P.bias_floats * 4 || ((uintptr_t)workspace & 127)) return B200ENV_EPARAMS;
    pa.n_layers = P.n_layers;
    pa.zs_off = P.zs_off;
    for (int l = 0; l < P.n_layers; ++l) pa.L[l] = P.L[l];
    pa.image = static_cast<unsigned char *>(workspace);
    pa.bias = reinterpret_cast<float *>(pa.image + img);
    policy_pack16_kernel<<<dim3(8, P.n_layers), 256, 0, stream>>>(pa);
    return b200_check_launch();
}

int policy_launch_umma16(int64_t n, const b200_mlp *actor, const b200_mlp *critic, const void *workspace, size_t bytes,
                         const PolicyIO &io, cudaStream_t stream) {
    HArgs a = {};
    int rc = h_build_plan(actor, critic, &a.p, nullptr, nullptr);
    if (rc) return rc;
    const size_t img = (size_t)(a.p.img_bytes + 127) / 128 * 128;
    if (!workspace) return B200ENV_ENULL;
    if (bytes < img + (size_t)a.p.bias_floats * 4 || ((uintptr_t)workspace & 127)) return B200ENV_EPARAMS;
    a.image = static_cast<const unsigned char *>(workspace);
    a.bias = reinterpret_cast<const float *>(a.image + img);
    a.io = io;
    static size_t configured[64] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) dev = 0;
    if (a.p.smem_bytes > configured[dev]) {
        if (cudaFuncSetAttribute(policy_umma16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)H_SMEM_LIMIT) != cudaSuccess)
            return b200_check_launch();
        configured[dev] = H_SMEM_LIMIT;
    }
    const int64_t tiles = (n + H_TILE - 1) / H_TILE, groups = (tiles + H_SLOTS - 1) / H_SLOTS;
    const unsigned cap = b200_persistent_grid(n, 1, 1);
    const unsigned grid = (unsigned)(groups < (int64_t)cap ? groups : (int64_t)cap);
    policy_umma16_kernel<<<grid, H_THREADS, a.p.smem_bytes, stream>>>(a, n);
    return b200_check_launch();
}
