// common.cuh -- shared device helpers of the batched environment kernels.
//
// One thread owns one environment instance; all per-instance arrays are
// field-major SoA ([field][n]) so that consecutive threads touch consecutive
// addresses (fully coalesced 8 B / 4 B accesses).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include "../../include/b200env.h"
#include "fastmath64.cuh"

#define B200_BLOCK 128

// ---------------------------------------------------------------------------
// Math traits: the fp64 path uses the libdevice double routines (1-2 ulp), the
// fp32 path the float ones.  No fast-math intrinsics: the fp32 tolerance is
// stated per env in the tests.
// ---------------------------------------------------------------------------
template <typename T> struct Mth;

template <> struct Mth<double> {
#ifdef B200_LIBDEVICE_MATH // A/B switch: libdevice everywhere
    static __device__ __forceinline__ void sincos(double x, double *s, double *c) { ::sincos(x, s, c); }
    static __device__ __forceinline__ void sincos3(double a, double b, double c, double *sa, double *ca, double *sb,
                                                   double *cb, double *sc, double *cc) {
        ::sincos(a, sa, ca); ::sincos(b, sb, cb); ::sincos(c, sc, cc);
    }
    static __device__ __forceinline__ void sincos2(double a, double b, double *sa, double *ca, double *sb, double *cb) {
        ::sincos(a, sa, ca); ::sincos(b, sb, cb);
    }
    static __device__ __forceinline__ double rcp(double y) { return 1.0 / y; }
    static __device__ __forceinline__ double div(double x, double y) { return x / y; }
    static __device__ __forceinline__ double tanh(double x) { return ::tanh(x); }
    static __device__ __forceinline__ double log(double x) { return ::log(x); }
    static __device__ __forceinline__ double log_nonneg(double x) { return ::log(x); }
    static __device__ __forceinline__ double exp(double x) { return ::exp(x); }
    static __device__ __forceinline__ double asin(double x) { return ::asin(x); }
#else // fastmath64.cuh: constant-bank coefficients, no special-case ladders, ~1 ulp
    static __device__ __forceinline__ void sincos(double x, double *s, double *c) { fm64::sincos(x, s, c); }
    static __device__ __forceinline__ void sincos3(double a, double b, double c, double *sa, double *ca, double *sb,
                                                   double *cb, double *sc, double *cc) {
        fm64::sincos3(a, b, c, sa, ca, sb, cb, sc, cc);
    }
    static __device__ __forceinline__ void sincos2(double a, double b, double *sa, double *ca, double *sb, double *cb) {
        fm64::sincos2(a, b, sa, ca, sb, cb);
    }
    static __device__ __forceinline__ double rcp(double y) { return fm64::rcp(y); }
    static __device__ __forceinline__ double div(double x, double y) { return fm64::div(x, y); }
    static __device__ __forceinline__ double tanh(double x) { return fm64::tanh(x); }
    static __device__ __forceinline__ double log(double x) { return fm64::log(x); }
    static __device__ __forceinline__ double log_nonneg(double x) { return fm64::log_nonneg(x); }
    static __device__ __forceinline__ double exp(double x) { return fm64::exp(x); }
    static __device__ __forceinline__ double asin(double x) { return fm64::asin(x); }
#endif
#ifndef B200_LIBDEVICE_MATH // a lone sin / cos also goes through the constant-bank sincos kernels: libdevice's versions
                            // were half of K-BB's instructions (+11 % there, +14 % on K-FASD)
    static __device__ __forceinline__ double sin(double x) { double s, c; fm64::sincos(x, &s, &c); return s; }
    static __device__ __forceinline__ double cos(double x) { double s, c; fm64::sincos(x, &s, &c); return c; }
#else
    static __device__ __forceinline__ double sin(double x) { return ::sin(x); }
    static __device__ __forceinline__ double cos(double x) { return ::cos(x); }
#endif
    static __device__ __forceinline__ double sin_ld(double x) { return ::sin(x); } // libdevice: faster where only sin is needed twice (K-TLM, A/B)
    static __device__ __forceinline__ double tan(double x) { return ::tan(x); }
    static __device__ __forceinline__ double pow(double x, double y) { return ::pow(x, y); }
    static __device__ __forceinline__ double sqrt(double x) { return ::sqrt(x); }
    static __device__ __forceinline__ double acos(double x) { return ::acos(x); }
    static __device__ __forceinline__ double atan2(double y, double x) { return ::atan2(y, x); }
    static __device__ __forceinline__ double abs(double x) { return ::fabs(x); }
    static __device__ __forceinline__ double min(double a, double b) { return ::fmin(a, b); }
    static __device__ __forceinline__ double max(double a, double b) { return ::fmax(a, b); }
    static __device__ __forceinline__ double fma(double a, double b, double c) { return ::fma(a, b, c); }
};

template <> struct Mth<float> {
    static __device__ __forceinline__ float sin(float x) { return ::sinf(x); }
    static __device__ __forceinline__ float sin_ld(float x) { return ::sinf(x); }
    static __device__ __forceinline__ float cos(float x) { return ::cosf(x); }
    static __device__ __forceinline__ void sincos(float x, float *s, float *c) { ::sincosf(x, s, c); }
    static __device__ __forceinline__ void sincos3(float a, float b, float c, float *sa, float *ca, float *sb, float *cb,
                                                   float *sc, float *cc) {
        ::sincosf(a, sa, ca); ::sincosf(b, sb, cb); ::sincosf(c, sc, cc);
    }
    static __device__ __forceinline__ void sincos2(float a, float b, float *sa, float *ca, float *sb, float *cb) {
        ::sincosf(a, sa, ca); ::sincosf(b, sb, cb);
    }
    static __device__ __forceinline__ float rcp(float y) { return 1.0f / y; }
    static __device__ __forceinline__ float div(float x, float y) { return x / y; }
    static __device__ __forceinline__ float tan(float x) { return ::tanf(x); }
    static __device__ __forceinline__ float tanh(float x) { return ::tanhf(x); }
    static __device__ __forceinline__ float pow(float x, float y) { return ::powf(x, y); }
    static __device__ __forceinline__ float log(float x) { return ::logf(x); }
    static __device__ __forceinline__ float log_nonneg(float x) { return ::logf(x); }
    static __device__ __forceinline__ float exp(float x) { return ::expf(x); }
    static __device__ __forceinline__ float sqrt(float x) { return ::sqrtf(x); }
    static __device__ __forceinline__ float asin(float x) { return ::asinf(x); }
    static __device__ __forceinline__ float acos(float x) { return ::acosf(x); }
    static __device__ __forceinline__ float atan2(float y, float x) { return ::atan2f(y, x); }
    static __device__ __forceinline__ float abs(float x) { return ::fabsf(x); }
    static __device__ __forceinline__ float min(float a, float b) { return ::fminf(a, b); }
    static __device__ __forceinline__ float max(float a, float b) { return ::fmaxf(a, b); }
    static __device__ __forceinline__ float fma(float a, float b, float c) { return ::fmaf(a, b, c); }
};

// x^a for x >= 0 given L = log(x): exp(a * L), with pow()'s conventions x^0 = 1 and 0^a = 0 (a > 0), inf (a < 0).
// Sharing L between |e|^alpha and |e|^(alpha-1) replaces two libdevice pow() calls (165 instructions each, measured
// with ncu) by one log and two exp.  Relative error <= (|a L| + 1) ulp, i.e. ~4e-15 for |a L| <= 35.
template <typename T>
__device__ __forceinline__ T pow_from_log(T L, T a) {
    const T r = Mth<T>::exp(a * L); // evaluated unconditionally: a select instead of a branch
    return a == (T)0 ? (T)1 : r;
}

// I/O-side accessors (action, dis in; obs, next_obs, reward, reset_obs out).  IO32 = the buffers hold float32 although
// the kernel computes in T = double (b200env_io::io_dtype == B200ENV_F32): the RL side of the reference is float32
// (actor output, RolloutBuffer.to_tensor utils/classes.py:292-301), so float32 I/O halves the PCIe / HBM bytes of the
// interface without touching the fp64 trajectory.  float -> double is exact; outputs are rounded once on store.
// Addressing of element (field, i) of a field-major [fields][n] buffer.  Default: byte address = base + i * ES + n *
// (field * ES) with i and n taken as 32-bit values (b200env_* rejects n >= 2^31: no env fits more instances in 180 GB)
// -- two IMAD.WIDE.U32, the second with an immediate multiplier, and the first is common to all fields of a buffer.
// The index form `base[field * n + i]` cost ~8 instructions per access in the UAV kernels (ncu source page: 15 % of all
// executed instructions); switching gave +18 % on K-UAVP and +16 % on K-UAVA.  B200_SOA_INDEX (defined by ugvo.cu,
// whose warp-cooperative kernel gets slower with the extra live pointer pairs) keeps the index form.
#ifndef B200_SOA_INDEX
template <typename T, bool IO32, typename I>
__device__ __forceinline__ T ldio(const void *base, I n, int field, I i) {
    constexpr int ES = IO32 ? 4 : (int)sizeof(T);
    const char *p = static_cast<const char *>(base) + (uint64_t)(uint32_t)i * ES + (uint64_t)(uint32_t)n * (uint32_t)(field * ES);
    if (IO32) return (T) * reinterpret_cast<const float *>(p);
    return *reinterpret_cast<const T *>(p);
}
template <typename T, bool IO32, typename I>
__device__ __forceinline__ void stio(void *base, I n, int field, I i, T v) {
    constexpr int ES = IO32 ? 4 : (int)sizeof(T);
    char *p = static_cast<char *>(base) + (uint64_t)(uint32_t)i * ES + (uint64_t)(uint32_t)n * (uint32_t)(field * ES);
    if (IO32) *reinterpret_cast<float *>(p) = (float)v;
    else *reinterpret_cast<T *>(p) = v;
}
#else
template <typename T, bool IO32, typename I>
__device__ __forceinline__ T ldio(const void *base, I n, int field, I i) {
    if (IO32) return (T) static_cast<const float *>(base)[(I)field * n + i];
    return static_cast<const T *>(base)[(I)field * n + i];
}
template <typename T, bool IO32, typename I>
__device__ __forceinline__ void stio(void *base, I n, int field, I i, T v) {
    if (IO32) static_cast<float *>(base)[(I)field * n + i] = (float)v;
    else static_cast<T *>(base)[(I)field * n + i] = v;
}
#endif

// Division by a quantity that is fixed over many quotients.  One IEEE reciprocal r = RN(1 / d), then per quotient
// q = a r and one FMA-corrected Newton step q + (a - q d) r (Markstein): 3 instructions instead of the ~25 of an fp64
// division.  The corrected quotient is the IEEE quotient except in rare half-way cases (<= 1 ulp there), far inside
// the 1e-12 parity bar; NaN / inf numerators propagate.  The RK4 updates of every reference env divide by 6
// (`(K1 + 2 K2 + 2 K3 + K4) / 6`), the time-loop envs 40+ times per control period.
// index-form I/O accessors, always available: the fused multi-step kernel (env_kernel.cuh) walks time-major rows whose
// base pointer changes every step, where `row[field * n + i]` is cheaper than re-deriving the pointer form (SOI rollout:
// 4.85 ms vs 6.25 ms for 2048 x 131072 steps)
template <typename T, bool IO32, typename I>
__device__ __forceinline__ T ldio_idx(const void *base, I n, int field, I i) {
    if (IO32) return (T) static_cast<const float *>(base)[(I)field * n + i];
    return static_cast<const T *>(base)[(I)field * n + i];
}
template <typename T, bool IO32, typename I>
__device__ __forceinline__ void stio_idx(void *base, I n, int field, I i, T v) {
    if (IO32) static_cast<float *>(base)[(I)field * n + i] = (float)v;
    else static_cast<T *>(base)[(I)field * n + i] = v;
}

// np.linalg.norm of a 2-vector (a, b) as the reference's numpy evaluates it: sqrt(x.dot(x)) with OpenBLAS' ddot, whose
// accumulation is FMA-contracted -- sqrt(fma(b, b, a * a)), not sqrt(a * a + b * b).  Pinned by the collision-radius-equality
// fixture tests/golden/ugvo_edge.npz (the plain form flips 2 of 180 `distance <= r + r_vehicle` decisions) and by
// SecondOrderIntegration's reward, which is bit-exact only with this form (oracle/c/small_envs.c).
template <typename T>
__device__ __forceinline__ T np_norm2(T a, T b) { return Mth<T>::sqrt(Mth<T>::fma(b, b, a * a)); }

// Sum of squares a^2 + b^2 (+ c^2 + d^2), left to right with every product and sum rounded on its own, as a Python
// expression `a * a + b * b + ...` evaluates it.  The _rn intrinsics are never contracted into FMAs, so the result does
// not depend on -fmad: a decision such as CartPole's `sqrt(...) < 1e-2` then takes the reference's side at the threshold
// (contracted, it flips in a few percent of the states within an ulp of it; tests/test_env_edges_gpu.py).
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
template <typename T>
__device__ __forceinline__ T sumsq_rn(T a, T b) { return add_rn(mul_rn(a, a), mul_rn(b, b)); }
template <typename T>
__device__ __forceinline__ T sumsq_rn(T a, T b, T c, T d) {
    return add_rn(add_rn(sumsq_rn(a, b), mul_rn(c, c)), mul_rn(d, d));
}

// clamp against bounds that are never NaN: two compare-selects instead of the NaN-aware fmin / fmax pair (6 instructions
// each in fp64).  A NaN x passes through, like np.clip.
template <typename T>
__device__ __forceinline__ T clampc(T x, T lo, T hi) {
    x = x < lo ? lo : x;
    return x > hi ? hi : x;
}

template <typename T>
struct Divisor {
    T d, r;
    __device__ __forceinline__ explicit Divisor(T d_) : d(d_), r((T)1 / d_) {}
    // reciprocal supplied by the caller: a host-side 1 / d, or Mth<T>::rcp(d) (<= 1 ulp) where the divisor changes per
    // thread -- the compiler's IEEE division costs ~25 instructions and a slow-path branch that splits the basic block
    __device__ __forceinline__ Divisor(T d_, T r_) : d(d_), r(r_) {}
    __device__ __forceinline__ T div(T a) const {
        const T q = a * r;
        return Mth<T>::fma(Mth<T>::fma(-q, d, a), r, q);
    }
};
template <typename T>
__device__ __forceinline__ T div6(T a) {
    const T r = (T)(1.0 / 6.0);
    const T q = a * r;
    return Mth<T>::fma(Mth<T>::fma(-q, (T)6, a), r, q);
}

// ---------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11).  Counter = (env index lo, env index hi,
// episode, block); key = 64-bit seed.  Results are therefore independent of
// the launch geometry and of how instances are sharded over GPUs.
// ---------------------------------------------------------------------------
struct Philox {
    uint32_t c0, c1, c2, c3; // counter
    uint32_t k0, k1;         // key
    uint32_t r[4];           // last block
    int have;                // unread words in r

    __device__ __forceinline__ Philox(uint64_t seed, uint64_t env, uint32_t episode)
        : c0((uint32_t)env), c1((uint32_t)(env >> 32)), c2(episode), c3(0u),
          k0((uint32_t)seed), k1((uint32_t)(seed >> 32)), have(0) {}

    __device__ __forceinline__ void block() {
        uint32_t x0 = c0, x1 = c1, x2 = c2, x3 = c3, ka = k0, kb = k1;
#pragma unroll
        for (int i = 0; i < 10; ++i) {
            const uint32_t hi0 = __umulhi(0xD2511F53u, x0), lo0 = 0xD2511F53u * x0;
            const uint32_t hi1 = __umulhi(0xCD9E8D57u, x2), lo1 = 0xCD9E8D57u * x2;
            const uint32_t y0 = hi1 ^ x1 ^ ka, y1 = lo1, y2 = hi0 ^ x3 ^ kb, y3 = lo0;
            x0 = y0; x1 = y1; x2 = y2; x3 = y3;
            ka += 0x9E3779B9u; kb += 0xBB67AE85u;
        }
        r[0] = x0; r[1] = x1; r[2] = x2; r[3] = x3;
        ++c3;
        have = 4;
    }

    // uniform double in [0,1) with 53 random bits (two 32-bit words)
    __device__ __forceinline__ double u01() {
        if (have < 2) block();
        const uint32_t a = r[4 - have], b = r[5 - have];
        have -= 2;
        return ((double)(a >> 5) * 67108864.0 + (double)(b >> 6)) * (1.0 / 9007199254740992.0);
    }

    // U(lo, hi) = fma(hi - lo, u, lo): one rounding, reproducible on the CPU with fma()
    __device__ __forceinline__ double uniform(double lo, double hi) { return ::fma(hi - lo, u01(), lo); }
};

// ---------------------------------------------------------------------------
// SoA accessors
// ---------------------------------------------------------------------------
// The index type I is int64_t in general; the hot UAV kernels are also instantiated with uint32_t (chosen by the
// launcher when fields * n < 2^32), which turns ~5 instructions of 64-bit address arithmetic per access into
// IMAD + IMAD.WIDE.U32 (8 % of the executed instructions of the UAV-pos step, ncu).
#ifndef B200_SOA_INDEX
template <typename T, typename I>
__device__ __forceinline__ T ld(const void *base, I n, int field, I i) {
    const char *bi = static_cast<const char *>(base) + (uint64_t)(uint32_t)i * sizeof(T);
    return *reinterpret_cast<const T *>(bi + (uint64_t)(uint32_t)n * (uint32_t)(field * (int)sizeof(T)));
}
template <typename T, typename I>
__device__ __forceinline__ void st(void *base, I n, int field, I i, T v) {
    char *bi = static_cast<char *>(base) + (uint64_t)(uint32_t)i * sizeof(T);
    *reinterpret_cast<T *>(bi + (uint64_t)(uint32_t)n * (uint32_t)(field * (int)sizeof(T))) = v;
}
#else
template <typename T, typename I>
__device__ __forceinline__ T ld(const void *base, I n, int field, I i) {
    return static_cast<const T *>(base)[(I)field * n + i];
}
template <typename T, typename I>
__device__ __forceinline__ void st(void *base, I n, int field, I i, T v) {
    static_cast<T *>(base)[(I)field * n + i] = v;
}
#endif

// ---------------------------------------------------------------------------
// host-side launch helpers
// ---------------------------------------------------------------------------
extern thread_local int g_b200_last_cuda_error;

static inline int b200_check_launch() {
    cudaError_t e = cudaPeekAtLastError();
    if (e != cudaSuccess) {
        g_b200_last_cuda_error = (int)e;
        cudaGetLastError(); // clear the non-sticky error
        return B200ENV_ECUDA;
    }
    return B200ENV_OK;
}

// number of SMs of the current device (148 on B200), queried once per device
static inline int b200_sm_count() {
    static int sms[64] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) dev = 0;
    if (!sms[dev]) {
        int v = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
        sms[dev] = v;
    }
    return sms[dev];
}

// grid of a persistent kernel: blocks_per_sm resident blocks on every SM of the current device, never more blocks than
// tiles
static inline unsigned b200_persistent_grid(int64_t n, int blocks_per_sm, int block = B200_BLOCK) {
    const int64_t tiles = (n + block - 1) / block, cap = (int64_t)b200_sm_count() * blocks_per_sm;
    return (unsigned)(tiles < cap ? tiles : cap);
}

// raises `kernel`'s dynamic shared-memory limit to `bytes` where a launch needs more than the default 48 KB, once per
// device and size (configured: the kernel's limit so far, per device)
template <typename Kernel>
static inline int b200_opt_in_smem(Kernel kernel, size_t bytes, size_t (&configured)[64]) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 64) dev = 0;
    if (bytes > 48 * 1024 && bytes > configured[dev]) {
        if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess)
            return b200_check_launch();
        configured[dev] = bytes;
    }
    return B200ENV_OK;
}
// float32 I/O buffers with fp64 arithmetic (b200env_io::io_dtype); in F32 mode everything is float anyway
static inline bool b200_io32(const b200env_io *io) { return io->io_dtype == B200ENV_F32; }
// launches KERN<T, IO32> for (double, io32) / (double, native) / float; expects `dtype` and `io` in scope
#define B200_LAUNCH_TIO(KERN, grid, block, s, ...)                                                                   \
    do {                                                                                                             \
        if (dtype == B200ENV_F64 && b200_io32(io)) KERN<double, true><<<grid, block, 0, s>>>(__VA_ARGS__);           \
        else if (dtype == B200ENV_F64) KERN<double, false><<<grid, block, 0, s>>>(__VA_ARGS__);                      \
        else KERN<float, false><<<grid, block, 0, s>>>(__VA_ARGS__);                                                 \
    } while (0)
static inline unsigned b200_grid(int64_t n, int block = B200_BLOCK) { return (unsigned)((n + block - 1) / block); }

// per-family entry points (defined in the family's .cu file)
#define B200_FAMILY_DECL(name)                                                                                  \
    int name##_dims(int variant, int *sf, int *od, int *ad, int *dd);                                           \
    int name##_step(int dtype, int64_t n, const void *params, const b200env_io *io, uint32_t flags,              \
                    uint64_t seed, int64_t off, cudaStream_t s);                                                \
    int name##_reset(int dtype, int64_t n, const void *params, const b200env_io *io, const uint8_t *mask,        \
                     uint64_t seed, int64_t off, cudaStream_t s);                                               \
    int name##_observe(int dtype, int64_t n, const void *params, const b200env_io *io, cudaStream_t s);

B200_FAMILY_DECL(cartpole)
B200_FAMILY_DECL(uav_att)
B200_FAMILY_DECL(uav_pos)
B200_FAMILY_DECL(fas)
B200_FAMILY_DECL(soi)
B200_FAMILY_DECL(ballbalancer)
B200_FAMILY_DECL(twolink)
B200_FAMILY_DECL(ugv)
B200_FAMILY_DECL(ugvo)
B200_FAMILY_DECL(uavrobust)
B200_FAMILY_DECL(fas_discrete)
// families built on env_kernel.cuh also have a fused multi-step kernel (state in registers across the steps)
#define B200_FAMILY_ROLLOUT_DECL(name)                                                                          \
    int name##_rollout(int dtype, int64_t n, const void *params, const b200env_io *io,                          \
                       const b200env_rollout_spec *rs, uint32_t flags, uint64_t seed, int64_t off, cudaStream_t s);
B200_FAMILY_ROLLOUT_DECL(cartpole)
B200_FAMILY_ROLLOUT_DECL(fas)
B200_FAMILY_ROLLOUT_DECL(soi)
B200_FAMILY_ROLLOUT_DECL(ballbalancer)
B200_FAMILY_ROLLOUT_DECL(twolink)
B200_FAMILY_ROLLOUT_DECL(ugv)
B200_FAMILY_ROLLOUT_DECL(fas_discrete)
