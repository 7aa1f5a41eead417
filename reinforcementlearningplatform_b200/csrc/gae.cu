// gae.cu -- K-GAE: PPO2 / DPPO2 generalised-advantage reverse scan over a time-major [T, N] rollout (sm_100a).
//
// Replaces the Python loop of algorithm/policy_base/Proximal_Policy_Optimization2.py:88-100 (and the identical
// Worker.learn lines of Distributed_PPO2.py:59-71):
//     deltas   = r + gamma * (1 - success) * V(s') - V(s)                   float32 tensors
//     gae_t    = delta_t + gamma * lmd * gae_{t+1} * (1 - done_t)           reverse loop, gae_T = 0
//     v_target = adv + V(s);   adv <- (adv - mean) / (std_unbiased + 1e-5)
// The reference holds one env (N = 1, T = buffer size); here every column n of the [T, N] arrays is one env instance,
// one thread walks its column backwards, and consecutive threads read consecutive addresses (28 B of HBM traffic per
// element: 5 float loads + 2 float stores).
//
// Exactness: with acc_mode 0 every operation is a separately rounded float32 multiply/add (__fmul_rn/__fadd_rn, no
// FMA contraction) in the reference's evaluation order, i.e. bit-identical to the loop under numpy >= 2 (NEP 50:
// python floats are weak, the scan runs in float32).  acc_mode 1 carries gae in float64 (the numpy 1.x behaviour).
// The per-launch (sum adv, sum adv^2, count) are accumulated in float64: every block writes its two partial sums to a
// caller-owned scratch array and a one-block kernel adds them up in a fixed order (strided per-thread sums, then a fixed
// tree) before incrementing stats[3] -- the same bits on every run, like K-NORM's statistics; ready for a 3-double
// all-reduce when the rollout is sharded over GPUs (global advantage normalisation).  Without scratch the partial sums
// fall back to atomicAdd (order-dependent in the last bits).
#include "common.cuh"

namespace {

constexpr int GAE_BLOCK = 128;
constexpr int GAE_UNROLL = 4;

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    return v;
}

// per-block part of the (sum, sum of squares, count) statistics: warp sums, then the block's warps in order; thread 0
// writes the block's two partials to scratch (partial[2 b], partial[2 b + 1], added up by gae_stats_reduce_kernel) or,
// without scratch, adds them atomically
template <int WARPS>
__device__ __forceinline__ void block_stats(double s1, double s2, int64_t T, int64_t N, double *stats, double *partial) {
    __shared__ double sh1[WARPS], sh2[WARPS];
    s1 = warp_sum(s1);
    s2 = warp_sum(s2);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (lane == 0) { sh1[w] = s1; sh2[w] = s2; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0, b = 0;
#pragma unroll
        for (int k = 0; k < WARPS; ++k) { a += sh1[k]; b += sh2[k]; }
        if (partial) {                      // deterministic path: block b owns partial[2 b], partial[2 b + 1]
            partial[2 * (int64_t)blockIdx.x] = a;
            partial[2 * (int64_t)blockIdx.x + 1] = b;
        } else {
            atomicAdd(stats + 0, a);
            atomicAdd(stats + 1, b);
            if (blockIdx.x == 0) atomicAdd(stats + 2, (double)T * (double)N);
        }
    }
}

// how the two masks of the scan are stored: FloatMasks = the reference's float32 `done` / `success` columns
// (RolloutBuffer.to_tensor, utils/classes.py:292-301); FlagMasks = what the step kernels write into a device-resident
// rollout (rollout.py): `done` as u8 and the terminal flag as i32, with success = done && flag != timeout_flag -- the
// rule of the train loops (PPO2-4-CartPoleAngleOnly/train.py:198-205, PPO2-4-UavFntsmcParamPos/train.py:299-302).
struct FloatMasks {
    const float *done, *succ;
    __device__ __forceinline__ void load(int64_t idx, float &d, float &s) const { d = __ldcs(done + idx); s = __ldcs(succ + idx); }
};
struct FlagMasks {
    const uint8_t *done;
    const int32_t *flag;
    int32_t timeout_flag;
    __device__ __forceinline__ void load(int64_t idx, float &d, float &s) const {
        const bool dn = __ldcs(done + idx) != 0;
        const int32_t f = __ldcs(flag + idx);
        d = dn ? 1.0f : 0.0f;
        s = (dn && f != timeout_flag) ? 1.0f : 0.0f;
    }
};

template <bool F64_ACC, class Masks>
__global__ void __launch_bounds__(GAE_BLOCK)
gae_kernel(int64_t T, int64_t N, const float *__restrict__ r, const float *__restrict__ vs,
           const float *__restrict__ vsn, const Masks mk, float g32,
           float gl32, double gl64, float *__restrict__ adv, float *__restrict__ vt, double *stats, double *partial) {
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double s1 = 0.0, s2 = 0.0;
    if (n < N) {
        float gae = 0.0f;
        double gae64 = 0.0;
        int64_t t = T - 1;
        // main loop: GAE_UNROLL time steps per trip, all loads of a trip issued before the dependent scan
        for (; t >= GAE_UNROLL - 1; t -= GAE_UNROLL) {
            float rr[GAE_UNROLL], v0[GAE_UNROLL], v1[GAE_UNROLL], dd[GAE_UNROLL], ss[GAE_UNROLL];
#pragma unroll
            for (int u = 0; u < GAE_UNROLL; ++u) {
                const int64_t idx = (t - u) * N + n;
                rr[u] = __ldcs(r + idx); v0[u] = __ldcs(vs + idx); v1[u] = __ldcs(vsn + idx);
                mk.load(idx, dd[u], ss[u]);
            }
#pragma unroll
            for (int u = 0; u < GAE_UNROLL; ++u) {
                const int64_t idx = (t - u) * N + n;
                // deltas = r + gamma * (1.0 - success) * vs_ - vs
                const float delta = __fsub_rn(__fadd_rn(rr[u], __fmul_rn(__fmul_rn(g32, __fsub_rn(1.0f, ss[u])), v1[u])), v0[u]);
                float a;
                if (F64_ACC) {
                    gae64 = (double)delta + gl64 * gae64 * (1.0 - (double)dd[u]);
                    a = (float)gae64;
                } else {
                    // gae = delta + gamma * lmd * gae * (1.0 - d)
                    gae = __fadd_rn(delta, __fmul_rn(__fmul_rn(gl32, gae), __fsub_rn(1.0f, dd[u])));
                    a = gae;
                }
                __stcs(adv + idx, a);
                __stcs(vt + idx, __fadd_rn(a, v0[u]));
                s1 += (double)a;
                s2 += (double)a * (double)a;
            }
        }
        for (; t >= 0; --t) {
            const int64_t idx = t * N + n;
            const float v0 = vs[idx];
            float dn, sc;
            mk.load(idx, dn, sc);
            const float delta = __fsub_rn(__fadd_rn(r[idx], __fmul_rn(__fmul_rn(g32, __fsub_rn(1.0f, sc)), vsn[idx])), v0);
            float a;
            if (F64_ACC) {
                gae64 = (double)delta + gl64 * gae64 * (1.0 - (double)dn);
                a = (float)gae64;
            } else {
                gae = __fadd_rn(delta, __fmul_rn(__fmul_rn(gl32, gae), __fsub_rn(1.0f, dn)));
                a = gae;
            }
            adv[idx] = a;
            vt[idx] = __fadd_rn(a, v0);
            s1 += (double)a;
            s2 += (double)a * (double)a;
        }
    }
    if (stats) block_stats<GAE_BLOCK / 32>(s1, s2, T, N, stats, partial);
}

// acc_mode 2: the same recurrence as a warp-level scan ALONG TIME, for rollouts with few columns (the reference's own
// shape is N = 1, T = 1000 .. 2048: one thread per column would walk 2048 dependent steps on one lane of one SM).  One
// warp owns a column; lane l of a trip holds time step hi - l with the affine map g -> b + a g (a = gamma lmd (1 - done),
// b = delta, delta rounded in float32 exactly like the reference); five shuffle steps compose the 32 maps (Kogge-Stone,
// the operator is associative), the carry g_{hi+1} enters at the end: T / 32 trips instead of T dependent steps.  The
// composition runs in float64, so the result is the float64-carry scan (acc_mode 1, numpy 1.x behaviour, note N12) up to
// float64 reassociation (~1e-15 relative), i.e. within one float32 ulp of it after the final rounding.
constexpr int SCAN_WARPS = 4;
template <class Masks>
__global__ void __launch_bounds__(SCAN_WARPS * 32)
gae_scan_kernel(int64_t T, int64_t N, const float *__restrict__ r, const float *__restrict__ vs,
                const float *__restrict__ vsn, const Masks mk, float g32, double gl64, float *__restrict__ adv,
                float *__restrict__ vt, double *stats, double *partial) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t n = (int64_t)blockIdx.x * SCAN_WARPS + w;
    double s1 = 0.0, s2 = 0.0;
    if (n < N) {
        double carry = 0.0;
        for (int64_t hi = T - 1; hi >= 0; hi -= 32) {
            const int64_t t = hi - lane;
            const bool valid = t >= 0;
            const int64_t idx = (valid ? t : 0) * N + n;
            const float v0 = vs[idx];
            float dn, sc;
            mk.load(idx, dn, sc);
            const float delta = __fsub_rn(__fadd_rn(r[idx], __fmul_rn(__fmul_rn(g32, __fsub_rn(1.0f, sc)), vsn[idx])), v0);
            double a = valid ? gl64 * (1.0 - (double)dn) : 1.0, b = valid ? (double)delta : 0.0;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {          // (a, b) of lanes 0 .. l composed: g(l) = b + a * g(-1)
                const double ap = __shfl_up_sync(0xffffffffu, a, o), bp = __shfl_up_sync(0xffffffffu, b, o);
                if (lane >= o) {
                    b = b + a * bp;
                    a = a * ap;
                }
            }
            const double g = b + a * carry;
            carry = __shfl_sync(0xffffffffu, g, 31);
            if (valid) {
                const float af = (float)g;
                adv[idx] = af;
                vt[idx] = __fadd_rn(af, v0);
                s1 += (double)af;
                s2 += (double)af * (double)af;
            }
        }
    }
    if (stats) {
        __shared__ double sh1[SCAN_WARPS], sh2[SCAN_WARPS];
        s1 = warp_sum(s1);
        s2 = warp_sum(s2);
        if (lane == 0) { sh1[w] = s1; sh2[w] = s2; }
        __syncthreads();
        if (threadIdx.x == 0) {
            double a = 0, b = 0;
#pragma unroll
            for (int k = 0; k < SCAN_WARPS; ++k) { a += sh1[k]; b += sh2[k]; }
            if (partial) {
                partial[2 * (int64_t)blockIdx.x] = a;
                partial[2 * (int64_t)blockIdx.x + 1] = b;
            } else {
                atomicAdd(stats + 0, a);
                atomicAdd(stats + 1, b);
                if (blockIdx.x == 0) atomicAdd(stats + 2, (double)T * (double)N);
            }
        }
    }
}

// fixed-order sum of the per-block partials: thread k adds partials k, k + 256, ... sequentially, then the 256 thread sums
// are combined by a fixed shared-memory tree; one thread increments stats
__global__ void __launch_bounds__(256) gae_stats_reduce_kernel(int64_t blocks, const double *__restrict__ partial,
                                                               double count, double *stats) {
    __shared__ double sh[2][256];
    double a = 0.0, b = 0.0;
    for (int64_t k = threadIdx.x; k < blocks; k += 256) {
        a += partial[2 * k];
        b += partial[2 * k + 1];
    }
    sh[0][threadIdx.x] = a;
    sh[1][threadIdx.x] = b;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) {
            sh[0][threadIdx.x] += sh[0][threadIdx.x + o];
            sh[1][threadIdx.x] += sh[1][threadIdx.x + o];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        stats[0] += sh[0][0];
        stats[1] += sh[1][0];
        stats[2] += count;
    }
}

// adv <- (adv - mean) / (std + eps), mean/std from (sum, sum of squares, count); unbiased std like torch.Tensor.std()
__global__ void __launch_bounds__(256)
adv_normalize_kernel(int64_t count, float *__restrict__ adv, const double *__restrict__ stats, double eps) {
    const double cnt = stats[2];
    const double mean = stats[0] / cnt;
    const double var = fmax((stats[1] - cnt * mean * mean) / (cnt - 1.0), 0.0);
    // (adv - adv.mean()) / (adv.std() + 1e-5) on float32 tensors: a true float32 division, like the reference
    const float m = (float)mean, den = __fadd_rn((float)sqrt(var), (float)eps);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x)
        adv[i] = __fdiv_rn(__fsub_rn(adv[i], m), den);
}

// PPO / DPPO (v1) Monte-Carlo return scan, SURVEY 8(f)-4: algorithm/policy_base/Proximal_Policy_Optimization.py:113-119,
// Distributed_PPO.py:58-64:
//     for reward, is_terminal in zip(reversed(buffer.r), reversed(buffer.done)):
//         if is_terminal: discounted_reward = 0
//         discounted_reward = reward + gamma * discounted_reward;  rewards.insert(0, discounted_reward)
//     rewards = torch.tensor(np.array(rewards), dtype=torch.float32)
// buffer.r is a float64 numpy array, so the recurrence runs in float64 (separately rounded multiply and add) and only
// the stored return is rounded to float32.  One thread per instance column, like K-GAE.
// STATS: the scan also sums the stored float32 returns and their squares in float64 and hands them to K-GAE's fixed-order
// reduction (block_stats into scratch, then gae_stats_reduce_kernel): the statistics of the v1 return normalisation.
// STATS = false is b200_mc_returns, instruction for instruction the kernel it was before the statistics existed.
template <typename TR, bool STATS>
__global__ void __launch_bounds__(GAE_BLOCK)
mc_returns_kernel(int64_t T, int64_t N, const TR *__restrict__ r, const uint8_t *__restrict__ done, double gamma,
                  float *__restrict__ ret, double *partial) {
    const int64_t n = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (!STATS && n >= N) return;
    double s1 = 0.0, s2 = 0.0;
    if (n < N) {
        double acc = 0.0;
        int64_t t = T - 1;
        constexpr int RET_UNROLL = 8;
        for (; t >= RET_UNROLL - 1; t -= RET_UNROLL) {
            double rr[RET_UNROLL];
            uint8_t dd[RET_UNROLL];
#pragma unroll
            for (int u = 0; u < RET_UNROLL; ++u) {
                const int64_t idx = (t - u) * N + n;
                rr[u] = (double)__ldcs(r + idx);
                dd[u] = __ldcs(done + idx);
            }
#pragma unroll
            for (int u = 0; u < RET_UNROLL; ++u) {
                if (dd[u]) acc = 0.0;
                acc = __dadd_rn(rr[u], __dmul_rn(gamma, acc));
                const float rf = (float)acc;
                __stcs(ret + (t - u) * N + n, rf);
                if (STATS) {
                    s1 += (double)rf;
                    s2 += (double)rf * (double)rf;
                }
            }
        }
        for (; t >= 0; --t) {
            const int64_t idx = t * N + n;
            if (done[idx]) acc = 0.0;
            acc = __dadd_rn((double)r[idx], __dmul_rn(gamma, acc));
            const float rf = (float)acc;
            ret[idx] = rf;
            if (STATS) {
                s1 += (double)rf;
                s2 += (double)rf * (double)rf;
            }
        }
    }
    if (STATS) block_stats<GAE_BLOCK / 32>(s1, s2, T, N, nullptr, partial);
}

} // namespace

namespace {
template <class Masks>
int gae_launch(int64_t T, int64_t N, const float *r, const float *vs, const float *vs_next, const Masks &mk, double gamma,
               double lmd, int acc_mode, float *adv, float *v_target, double *stats, void *scratch, size_t scratch_bytes,
               cudaStream_t s) {
    if (acc_mode < 0 || acc_mode > 2) return B200ENV_EPARAMS;
    const unsigned grid = acc_mode == 2 ? (unsigned)((N + SCAN_WARPS - 1) / SCAN_WARPS) : (unsigned)((N + GAE_BLOCK - 1) / GAE_BLOCK);
    const float g32 = (float)gamma, gl32 = (float)(gamma * lmd);
    double *partial = nullptr;
    if (stats && scratch) {
        if (scratch_bytes < (size_t)grid * 2 * sizeof(double) || ((uintptr_t)scratch & 7)) return B200ENV_EPARAMS;
        partial = static_cast<double *>(scratch);
    }
    if (acc_mode == 2)
        gae_scan_kernel<Masks><<<grid, SCAN_WARPS * 32, 0, s>>>(T, N, r, vs, vs_next, mk, g32, gamma * lmd, adv, v_target, stats, partial);
    else if (acc_mode == 0)
        gae_kernel<false, Masks><<<grid, GAE_BLOCK, 0, s>>>(T, N, r, vs, vs_next, mk, g32, gl32, gamma * lmd, adv, v_target, stats, partial);
    else
        gae_kernel<true, Masks><<<grid, GAE_BLOCK, 0, s>>>(T, N, r, vs, vs_next, mk, g32, gl32, gamma * lmd, adv, v_target, stats, partial);
    if (partial) gae_stats_reduce_kernel<<<1, 256, 0, s>>>((int64_t)grid, partial, (double)T * (double)N, stats);
    return b200_check_launch();
}
} // namespace

extern "C" B200_API size_t b200_gae_scratch_bytes(int64_t N) {
    return N <= 0 ? 0 : (size_t)((N + SCAN_WARPS - 1) / SCAN_WARPS) * 2 * sizeof(double);   // the finest grid (acc_mode 2)
}

extern "C" B200_API int b200_gae(int64_t T, int64_t N, const float *r, const float *vs, const float *vs_next,
                                 const float *done, const float *success, double gamma, double lmd, int acc_mode,
                                 float *adv, float *v_target, double *stats, void *scratch, size_t scratch_bytes,
                                 void *cuda_stream) {
    if (T <= 0 || N <= 0) return B200ENV_ESIZE;
    if (!r || !vs || !vs_next || !done || !success || !adv || !v_target) return B200ENV_ENULL;
    return gae_launch(T, N, r, vs, vs_next, FloatMasks{done, success}, gamma, lmd, acc_mode, adv, v_target, stats, scratch,
                      scratch_bytes, (cudaStream_t)cuda_stream);
}

extern "C" B200_API int b200_gae_flags(int64_t T, int64_t N, const float *r, const float *vs, const float *vs_next,
                                       const uint8_t *done, const int32_t *flag, int32_t timeout_flag, double gamma,
                                       double lmd, int acc_mode, float *adv, float *v_target, double *stats, void *scratch,
                                       size_t scratch_bytes, void *cuda_stream) {
    if (T <= 0 || N <= 0) return B200ENV_ESIZE;
    if (!r || !vs || !vs_next || !done || !flag || !adv || !v_target) return B200ENV_ENULL;
    return gae_launch(T, N, r, vs, vs_next, FlagMasks{done, flag, timeout_flag}, gamma, lmd, acc_mode, adv, v_target, stats,
                      scratch, scratch_bytes, (cudaStream_t)cuda_stream);
}

extern "C" B200_API int b200_adv_normalize(int64_t count, float *adv, const double *stats, double eps,
                                           void *cuda_stream) {
    if (count <= 0) return B200ENV_ESIZE;
    if (!adv || !stats) return B200ENV_ENULL;
    const int64_t cap = (int64_t)b200_sm_count() * 16;
    int64_t blocks = (count + 255) / 256;
    if (blocks > cap) blocks = cap;
    adv_normalize_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)cuda_stream>>>(count, adv, stats, eps);
    return b200_check_launch();
}

namespace {
int mc_returns_launch(int r_dtype, int64_t T, int64_t N, const void *r, const uint8_t *done, double gamma, float *returns,
                      double *stats, double *partial, cudaStream_t s) {
    const unsigned grid = (unsigned)((N + GAE_BLOCK - 1) / GAE_BLOCK);
    if (!stats) {
        if (r_dtype == B200ENV_F64) mc_returns_kernel<double, false><<<grid, GAE_BLOCK, 0, s>>>(T, N, (const double *)r, done, gamma, returns, nullptr);
        else mc_returns_kernel<float, false><<<grid, GAE_BLOCK, 0, s>>>(T, N, (const float *)r, done, gamma, returns, nullptr);
        return b200_check_launch();
    }
    if (r_dtype == B200ENV_F64) mc_returns_kernel<double, true><<<grid, GAE_BLOCK, 0, s>>>(T, N, (const double *)r, done, gamma, returns, partial);
    else mc_returns_kernel<float, true><<<grid, GAE_BLOCK, 0, s>>>(T, N, (const float *)r, done, gamma, returns, partial);
    gae_stats_reduce_kernel<<<1, 256, 0, s>>>((int64_t)grid, partial, (double)T * (double)N, stats);
    return b200_check_launch();
}
} // namespace

extern "C" B200_API int b200_mc_returns(int r_dtype, int64_t T, int64_t N, const void *r, const uint8_t *done,
                                        double gamma, float *returns, void *cuda_stream) {
    if (T <= 0 || N <= 0) return B200ENV_ESIZE;
    if (r_dtype != B200ENV_F64 && r_dtype != B200ENV_F32) return B200ENV_EDTYPE;
    if (!r || !done || !returns) return B200ENV_ENULL;
    return mc_returns_launch(r_dtype, T, N, r, done, gamma, returns, nullptr, nullptr, (cudaStream_t)cuda_stream);
}

extern "C" B200_API int b200_mc_returns_stats(int r_dtype, int64_t T, int64_t N, const void *r, const uint8_t *done,
                                              double gamma, float *returns, double *stats, void *scratch,
                                              size_t scratch_bytes, void *cuda_stream) {
    if (T <= 0 || N <= 0 || N >= ((int64_t)1 << 31)) return B200ENV_ESIZE;
    if (r_dtype != B200ENV_F64 && r_dtype != B200ENV_F32) return B200ENV_EDTYPE;
    if (!r || !done || !returns || !stats || !scratch) return B200ENV_ENULL;
    if (scratch_bytes < b200_gae_scratch_bytes(N) || ((uintptr_t)scratch & 7)) return B200ENV_EPARAMS;
    return mc_returns_launch(r_dtype, T, N, r, done, gamma, returns, stats, static_cast<double *>(scratch),
                             (cudaStream_t)cuda_stream);
}
