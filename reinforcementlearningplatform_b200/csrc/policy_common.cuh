// policy_common.cuh -- pieces shared by the K-POLICY kernels (policy.cu: FP32 FMA pipe; policy_umma.cu and
// policy_umma16.cu: tcgen05 tensor cores).
#pragma once
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
// policy_umma.cu (tcgen05 / TMEM): weights pre-packed into a caller-owned workspace
size_t policy_umma_workspace_bytes(const b200_mlp *actor, const b200_mlp *critic);
int policy_umma_pack(const b200_mlp *actor, const b200_mlp *critic, void *workspace, size_t bytes, cudaStream_t s);
int policy_launch_umma(int64_t n, const b200_mlp *actor, const b200_mlp *critic, const void *workspace, size_t bytes,
                       const PolicyIO &io, cudaStream_t s);
int policy_umma_probe(const float *A, const float *W, float *D, int N, int K, int three_pass, cudaStream_t s);
// policy_umma16.cu (tcgen05 / TMEM, fp16-split operands, four tiles in flight): the nets it holds (layers <= 64 wide,
// <= 32 observation fields) are routed to it by the three policy_umma_* entry points above
bool policy_umma16_fits(const b200_mlp *actor, const b200_mlp *critic);
size_t policy_umma16_workspace_bytes(const b200_mlp *actor, const b200_mlp *critic);
int policy_umma16_pack(const b200_mlp *actor, const b200_mlp *critic, void *workspace, size_t bytes, cudaStream_t s);
int policy_launch_umma16(int64_t n, const b200_mlp *actor, const b200_mlp *critic, const void *workspace, size_t bytes,
                         const PolicyIO &io, cudaStream_t s);

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
                act = fmaxf(fminf(act, amax), amin);
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
