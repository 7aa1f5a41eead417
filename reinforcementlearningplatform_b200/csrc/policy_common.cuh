// policy_common.cuh -- pieces shared by the K-POLICY kernels (policy.cu: FP32 FMA pipe; policy_umma.cu and
// policy_umma16.cu: tcgen05 tensor cores).
#pragma once
#include <cuda_fp16.h>
#include "common.cuh"

struct PolicyIO {
    const float *obs;            // [S][n]
    const float *a_min, *a_max;  // [A] device
    const float *noise;          // [A][n] or NULL
    const float *std_vec;        // [A] device per-dimension std (the DPPO2 demos' init_std = range / 6 vector), or NULL
    int out_affine;              // actor out_act == 2: mean = tanh(z) * gain + off, gain = a_max - off, off = (a_min + a_max) / 2
                                 // (demonstration/DPPO2/DPPO2-4-UGVForwardObstacleAvoidance/train.py:42-43,66-69)
    float std_;
    uint64_t seed, step;
    int64_t off;
    float *action, *log_prob, *mean, *value;
};

int policy_launch_fp32(int64_t n, const b200_mlp *actor, const b200_mlp *critic, const PolicyIO &io, cudaStream_t s);
int policy_umma_probe(const float *A, const float *W, float *D, int N, int K, int three_pass, cudaStream_t s);

// ------------------------------------------------------------------------------------------------ tcgen05 routes
// The two tcgen05 kernels (policy_umma16.cu for nets <= 64 wide with <= 32 observation fields, policy_umma.cu for the
// rest) read the same layer records, and their weights are packed by one kernel into a caller-owned workspace.
constexpr int POLICY_MAX_LAYERS = 8;

struct PolicyLayer {
    int K, N;        // padded: first layer K to a multiple of 8, others K = previous N; N to a multiple of 16
    int n_real;      // nn.Linear out features
    int role;        // 0 hidden (tanh), 1 actor output, 2 critic output
    int first;       // input = observations: 3xTF32 operand pairs, k-steps of 8
    int f16;         // operands as fp16 hi / lo pairs, weights pre-scaled by a power of two: k-steps of 16, half the
                     // image bytes and half the MMAs of the 3xTF32 form
    int out_act;     // output layers: 0 identity, 1 relu (2, the range map, is applied in policy_sample_store)
    uint32_t w_off;  // byte offset of the layer's image: k-step kk at w_off + kk * N * 64 (hi plane N * 32 B, then lo)
    int b_off;       // float offset of the layer's bias (tanh layers: pre-multiplied by 2 log2 e)
};

struct PolicyPlan {
    int n_layers, S, A;
    // policy_umma.cu's operating mode (build_plan); policy_umma16.cu has a single one and leaves these 0
    int slots, nbuf_log2, streamed;
    int a_tmem;      // 1: activations (A operand) live in TMEM and the MMAs are issued in the TS form; 0: shared memory (SS)
    int tmem_cols, slot_cols, pong_off, a_col;   // per slot: D ping at +0, D pong at +pong_off, A hi plane at +a_col,
                                                 // A lo plane at +a_col + 32 * nbuf (a_tmem only)
    uint32_t img_bytes;
    int bias_floats, zs_off;   // zs_off: per-layer accumulator scale (x 2 log2 e for tanh layers) inside the bias array
    uint32_t stage_bytes;
    uint32_t off_a, off_b, off_bias, off_scr, smem_bytes;  // dynamic shared memory map (after the barrier block)
    PolicyLayer L[POLICY_MAX_LAYERS];
};

// The kernel a net pair runs on, with its plan, and the nn.Linear weight / bias / in-features of every layer (for the
// packer; the actor's and the critic's input widths may differ, and only b200_policy_forward_packed rejects that)
struct PolicyRoute {
    PolicyPlan p;
    const float *w[POLICY_MAX_LAYERS], *b[POLICY_MAX_LAYERS];
    int k_real[POLICY_MAX_LAYERS];
    int (*launch)(int64_t n, const PolicyPlan &p, const PolicyIO &io, const unsigned char *image, const float *bias,
                  cudaStream_t s);
};

// Appends the layers of both nets to P->L and r->w / r->b / r->k_real, with their image and bias offsets: K padded to 8 on a net's
// first layer, N to 16.  The limits are the route's: layer width, first-layer input, and whether the layers after a
// net's first multiply fp16 pairs.  B200ENV_ESIZE for a net it does not hold.
int policy_add_nets(const b200_mlp *actor, const b200_mlp *critic, int max_width, int max_first_in, bool f16_hidden,
                    PolicyRoute *r);
// policy_umma16.cu's plan and launch when the pair fits it, else B200ENV_ESIZE
int policy_umma16_route(const b200_mlp *actor, const b200_mlp *critic, PolicyRoute *r);
// policy_umma16.cu when the pair fits it, else policy_umma.cu
int policy_route(const b200_mlp *actor, const b200_mlp *critic, PolicyRoute *r);
// weights and biases -> the workspace of the route, on the stream
int policy_pack(const PolicyRoute &r, void *workspace, size_t bytes, cudaStream_t s);

// The workspace of a plan: the weight image (rounded up to 128 bytes), then the bias floats
inline size_t policy_workspace_bytes(const PolicyPlan &p) {
    return ((size_t)p.img_bytes + 127) / 128 * 128 + (size_t)p.bias_floats * 4;
}
// a caller's workspace -> (image, bias); it must be 128-byte aligned and policy_workspace_bytes long
inline int policy_workspace_split(const PolicyPlan &p, void *workspace, size_t bytes, unsigned char **image, float **bias) {
    if (!workspace) return B200ENV_ENULL;
    if (bytes < policy_workspace_bytes(p) || ((uintptr_t)workspace & 127)) return B200ENV_EPARAMS;
    *image = static_cast<unsigned char *>(workspace);
    *bias = reinterpret_cast<float *>(*image + ((size_t)p.img_bytes + 127) / 128 * 128);
    return B200ENV_OK;
}

// eight values -> fp16 hi / lo pairs, hi = fp16(y), lo = fp16(y - hi) (22 significand bits, as a TF32 pair), two per
// word: the low half (.x) holds the even index
__device__ __forceinline__ void policy_split_f16x8(const float *y, uint32_t *hi, uint32_t *lo) {
#pragma unroll
    for (int p = 0; p < 4; ++p) {
        const __half2 h = __floats2half2_rn(y[2 * p], y[2 * p + 1]);
        const float2 f = __half22float2(h);
        const __half2 l = __floats2half2_rn(y[2 * p] - f.x, y[2 * p + 1] - f.y);
        hi[p] = *reinterpret_cast<const uint32_t *>(&h);
        lo[p] = *reinterpret_cast<const uint32_t *>(&l);
    }
}

// Philox key domain of the exploration noise.  The env resets draw from Philox(seed, instance, episode) (common.cuh); with
// equal seeds the reset of (instance i, episode e) and the noise of (instance i, step e) would consume the same 128-bit
// block, so the policy stream flips key bits the env stream never does ("POLI").
#define B200_POLICY_KEY_DOMAIN 0x504F4C49u

// Per-action-dimension constants of choose_action, [5][16] floats: a_min, a_max, std, log(std) + log(sqrt(2 pi)),
// 1 / (2 std^2).  Kernels that have shared memory to spare fill the table once per block (policy_dims_fill) instead of
// re-deriving log / reciprocal per instance and dimension.
#define B200_POLICY_DIMC_FLOATS 80
__device__ __forceinline__ void policy_dims_fill(const PolicyIO &a, int A, float *dimc, int tid, int nthreads) {
    for (int j = tid; j < 16; j += nthreads) {
        const bool on = j < A;
        const float sd = on ? (a.std_vec ? __ldg(a.std_vec + j) : a.std_) : 1.0f;
        dimc[j] = on ? __ldg(a.a_min + j) : 0.0f;
        dimc[16 + j] = on ? __ldg(a.a_max + j) : 0.0f;
        dimc[32 + j] = sd;
        dimc[48 + j] = logf(sd) + 0.91893853320467274178f;
        dimc[64 + j] = 1.0f / (2.0f * (sd * sd));
    }
}

// min / max that return NaN when either input is NaN (PTX min.NaN / max.NaN, sm_80+), one instruction like fminf / fmaxf,
// which would return the other input.  torch's choose_action turns a NaN observation into NaN outputs; with these the
// hidden-layer clamp, the relu head and the action clamp do too, instead of handing a diverged instance a plausible
// finite action.
__device__ __forceinline__ float policy_fmin_nan(float a, float b) {
    float d;
    asm("min.NaN.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b));
    return d;
}
__device__ __forceinline__ float policy_fmax_nan(float a, float b) {
    float d;
    asm("max.NaN.f32 %0, %1, %2;" : "=f"(d) : "f"(a), "f"(b));
    return d;
}

// tanh on the SFU (ex2.approx + rcp.approx), absolute error <= 4e-7: the range-mapped actor head
__device__ __forceinline__ float policy_tanh_sfu(float x) {
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * 2.885390081777927f));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
    return fmaf(-2.0f, r, 1.0f);
}

// Proximal_Policy_Optimization2.choose_action (:72-75) for instance i given its A means:
// a = clamp(mean + std * eps), log_prob = Normal(mean, std).log_prob(a).  eps: injected noise or Philox + Box-Muller.
// `mean_of(j)` returns the j-th pre-head output of instance i; `dimc`: the table above (shared memory) or NULL.
//
// Four action dimensions per pass = one Philox block = two Box-Muller pairs, written as straight-line code so that the
// four chains overlap: in the tcgen05 kernel one thread per instance runs this with one or two warps per scheduler, and
// round 1's two-at-a-time loop with libdevice logf / sqrtf / sincospif, a log(std) and an IEEE division per dimension
// took ~6500 cycles per tile (event trace, profiles/r2/policy_umma.md) -- more than the seven layers' epilogues.  The
// Gaussian draw now uses the SFU forms (lg2 / sqrt / sin / cos .approx: |error| ~1e-6 on a random number), the log-prob
// multiplies by 1 / (2 std^2) (<= 2 ulp from the reference's quotient).  Word k of block g still feeds dimension 4 g + k.
template <typename MeanFn>
__device__ __forceinline__ void policy_sample_store_fn(const PolicyIO &a, int64_t n, int64_t i, int A, MeanFn mean_of,
                                                       const float *dimc = nullptr) {
    Philox rng(a.seed, (uint64_t)(a.off + i), (uint32_t)a.step);
    rng.k1 ^= B200_POLICY_KEY_DOMAIN;
    rng.c3 = (uint32_t)(a.step >> 32) << 8; // high step bits above the block counter
    const float lstd0 = dimc ? 0.0f : logf(a.std_) + 0.91893853320467274178f;
    const float iv0 = dimc ? 0.0f : 1.0f / (2.0f * (a.std_ * a.std_));
    float *p_act = a.action + i, *p_lp = a.log_prob ? a.log_prob + i : nullptr, *p_mean = a.mean ? a.mean + i : nullptr;
    const float *p_noise = a.noise ? a.noise + i : nullptr;
    for (int j0 = 0; j0 < A; j0 += 4) {
        float e[4];
        if (p_noise) {
#pragma unroll
            for (int q = 0; q < 4; ++q) e[q] = j0 + q < A ? __ldcs(p_noise + (int64_t)q * n) : 0.0f;
            p_noise += 4 * n;
        } else { // Box-Muller on pairs of 32-bit uniforms; u1 in (0, 1]
            rng.block();
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const float u1 = ((float)(rng.r[2 * h] >> 8) + 1.0f) * (1.0f / 16777216.0f);
                const float ang = (float)(rng.r[2 * h + 1] >> 8) * (6.283185307179586f / 16777216.0f) - 3.14159265358979f;
                float l2, rad, sn, cs;
                asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(l2) : "f"(u1));
                asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(rad) : "f"(l2 * -1.3862943611198906f));   // sqrt(-2 ln u1)
                asm("sin.approx.ftz.f32 %0, %1;" : "=f"(sn) : "f"(ang));
                asm("cos.approx.ftz.f32 %0, %1;" : "=f"(cs) : "f"(ang));
                e[2 * h] = rad * cs;
                e[2 * h + 1] = rad * sn;
            }
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int j = j0 + q;
            if (j < A) {
                float m = mean_of(j);
                float amin, amax, sd, lstd, iv;
                if (dimc) {
                    amin = dimc[j]; amax = dimc[16 + j]; sd = dimc[32 + j]; lstd = dimc[48 + j]; iv = dimc[64 + j];
                } else {
                    amin = __ldg(a.a_min + j); amax = __ldg(a.a_max + j);
                    sd = a.std_; lstd = lstd0; iv = iv0;
                    if (a.std_vec) {
                        sd = __ldg(a.std_vec + j);
                        lstd = logf(sd) + 0.91893853320467274178f;
                        iv = 1.0f / (2.0f * (sd * sd));
                    }
                }
                if (a.out_affine) {
                    const float off = (amin + amax) / 2.0f;
                    m = policy_tanh_sfu(m) * (amax - off) + off;
                }
                float act = fmaf(sd, e[q], m);                                   // dist.sample()
                act = policy_fmax_nan(policy_fmin_nan(act, amax), amin);
                const float d = act - m;                                         // Normal.log_prob
                const float lp = -(d * d) * iv - lstd;
                __stcs(p_act + (int64_t)q * n, act);
                if (p_lp) __stcs(p_lp + (int64_t)q * n, lp);
                if (p_mean) __stcs(p_mean + (int64_t)q * n, m);
            }
        }
        p_act += 4 * n;
        if (p_lp) p_lp += 4 * n;
        if (p_mean) p_mean += 4 * n;
    }
}

__device__ __forceinline__ void policy_sample_store(const PolicyIO &a, int64_t n, int64_t i, int A, const float *src,
                                                    int stride, const float *dimc = nullptr) {
    policy_sample_store_fn(a, n, i, A, [src, stride](int j) { return src[j * stride]; }, dimc);
}
