// uav_common.cuh -- quadrotor dynamics, RK4, attitude kinematics and the FNTSMC laws shared by the UavFntsmcParam
// kernels (uav.cu) and the UavRobust kernels (uavrobust.cu).  Reference lines are cited at each function; the two
// families use the same maths (environment/UavRobust/uav.py:429-483 == environment/UavFntsmcParam/uav.py:93-148).
#pragma once
#include "common.cuh"

// ------------------------------------------------------------------------------------------------------------------
// B200_STRICT: the reference's operation order and library calls, one switch per shortcut of the shipped kernels, so that
// the free-running drift of the shipped build can be bounded and decomposed (tests/test_drift_gpu.py, `make strict`):
//   B200_STRICT_POW   |e|^alpha, |e|^(alpha-1), |s|^beta by three pow() calls      (shipped: one log + exp(a log x))
//   B200_STRICT_TAN   tan(theta) by tan()                                           (shipped: sin / cos)
//   B200_STRICT_DIV   IEEE divisions by J, m, cos(theta), cos^2(theta), 6, dt, 10   (shipped: reciprocal multiplies,
//                                                                                    Markstein-corrected quotients)
//   B200_UAV_LAPACK_INV  control = -inv(f1 h) (u1 + u2) by LU with partial pivoting (shipped: closed-form diag(J) f1^-1)
//   B200_LIBDEVICE_MATH  libdevice sincos / tanh / log / exp / asin                (shipped: fastmath64.cuh)
//   -fmad=false          no FMA contraction                                         (shipped: contraction on)
#ifdef B200_STRICT
#define B200_STRICT_POW
#define B200_STRICT_TAN
#define B200_STRICT_DIV
#ifndef B200_UAV_LAPACK_INV
#define B200_UAV_LAPACK_INV
#endif
#endif
#ifdef B200_STRICT_DIV
#define UAV_DIV(a, b, rb) ((a) / (b))
#else
#define UAV_DIV(a, b, rb) ((a) * (rb))
#endif

// Accessors of the persistent state buffer of the UAV families (UavFntsmcParam attitude / position, UavRobust):
// block-interleaved, element (field f,
// instance i) at [((i / 128) * B200_UAV_STATE_SLOTS + f) * 128 + i % 128] (include/b200env.h, b200env_state_layout).
// A thread's accesses to all fields are then ONE base register plus an immediate (f * 1024 B); with the field-major
// layout of the other buffers ([f][n], n a run-time value) every access needed its own IMAD.WIDE and a live 64-bit register
// pair: 144 -> 61 IMAD.WIDE in the position kernel, 0.220 -> 0.198 ms per 1 M instances (A/B on one box).  Coalescing is
// unchanged (128 consecutive doubles per field and block).  The `n` argument of the macros is unused; it keeps their
// call sites in the form of ld() / st() (common.cuh).
template <typename T, typename I>
__device__ __forceinline__ const char *uav_blk_base(const void *base, I i) {
    return static_cast<const char *>(base) +
           (uint64_t)((uint32_t)i >> 7) * (uint64_t)(B200_UAV_STATE_SLOTS * 128 * sizeof(T)) +
           ((uint32_t)i & 127u) * (uint32_t)sizeof(T);
}
#define UAV_LDS(base, n, field, i) (*reinterpret_cast<const T *>(uav_blk_base<T>(base, i) + (field) * (int)(128 * sizeof(T))))
#define UAV_STS(base, n, field, i, v) (*reinterpret_cast<T *>(const_cast<char *>(uav_blk_base<T>(base, i)) + (field) * (int)(128 * sizeof(T))) = (v))

namespace uavk {

typedef b200_uav_params P;



template <typename T>
struct Trig {
    T sphi, cphi, sth, cth, spsi, cpsi, tth, rcth;
    // one range check for all angles (fastmath64.cuh): the polynomial chains of the 2-3 sincos share a basic block
    __device__ __forceinline__ void eval(T phi, T th, T psi, bool need_psi) {
        if (need_psi) {
            Mth<T>::sincos3(phi, th, psi, &sphi, &cphi, &sth, &cth, &spsi, &cpsi);
        } else {
            Mth<T>::sincos2(phi, th, &sphi, &cphi, &sth, &cth);
            spsi = (T)0; cpsi = (T)1;
        }
        rcth = Mth<T>::rcp(cth);
#ifdef B200_STRICT_TAN
        tth = Mth<T>::tan(th);
#else
        tth = sth * rcth;
#endif
    }
};

// constants derived from the parameters on the HOST (launcher) and passed as a kernel argument: the reciprocals of
// J and m and kt / m used to be recomputed by every thread (five fp64 divisions, ~125 instructions per step)
struct UavDerived {
    double rJ[3], rm, kt_m, J21, J02, J10;
};
static inline UavDerived uav_derive(double m, const double *J, double kt) {
    UavDerived d;
    for (int k = 0; k < 3; ++k) d.rJ[k] = 1.0 / J[k];
    d.rm = 1.0 / m;
    d.kt_m = kt / m;
    d.J21 = J[2] - J[1]; d.J02 = J[0] - J[2]; d.J10 = J[1] - J[0];
    return d;
}

template <typename T>
struct Consts {
    T m, g, kr, kt, J0, J1, J2, J21, J02, J10, dt, rJ0, rJ1, rJ2, rm, kt_m;
    __device__ __forceinline__ Consts(double m_, double g_, const double *J, double kr_, double kt_, double dt_,
                                      const UavDerived &d)
        : m((T)m_), g((T)g_), kr((T)kr_), kt((T)kt_), J0((T)J[0]), J1((T)J[1]), J2((T)J[2]), J21((T)d.J21),
          J02((T)d.J02), J10((T)d.J10), dt((T)dt_), rJ0((T)d.rJ[0]), rJ1((T)d.rJ[1]), rJ2((T)d.rJ[2]), rm((T)d.rm),
          kt_m((T)d.kt_m) {}
};

// uav.py:93-124.  x = (x y z vx vy vz phi th psi p q r); only the derivative entries that the caller needs.
template <typename T, bool ATT_ONLY>
__device__ __forceinline__ void uav_ode(const Consts<T> &c, const T *x, const Trig<T> &t, T throttle, const T *tq,
                                        const T *dis, T *d) {
    const T p = x[9], q = x[10], r = x[11];
    // divisions by the constants J, m are multiplications by their reciprocals (<= 1 ulp from the reference's x / J)
    d[9] = UAV_DIV(-c.kr * p - q * r * c.J21 + tq[0], c.J0, c.rJ0);
    d[10] = UAV_DIV(-c.kr * q - p * r * c.J02 + tq[1], c.J1, c.rJ1);
    d[11] = UAV_DIV(-c.kr * r - p * q * c.J10 + tq[2], c.J2, c.rJ2);
    d[6] = p + (t.tth * t.sphi) * q + (t.tth * t.cphi) * r;
    d[7] = t.cphi * q - t.sphi * r;
    d[8] = UAV_DIV(t.sphi, t.cth, t.rcth) * q + UAV_DIV(t.cphi, t.cth, t.rcth) * r;
    if (!ATT_ONLY) {
        d[0] = x[3]; d[1] = x[4]; d[2] = x[5];
        d[3] = UAV_DIV(throttle * (t.cpsi * t.sth * t.cphi + t.spsi * t.sphi) - c.kt * x[3] + dis[0], c.m, c.rm);
        d[4] = UAV_DIV(throttle * (t.spsi * t.sth * t.cphi - t.cpsi * t.sphi) - c.kt * x[4] + dis[1], c.m, c.rm);
        d[5] = -c.g + UAV_DIV(throttle * t.cphi * t.cth - c.kt * x[5] + dis[2], c.m, c.rm);
    }
}

// uav.py:126-148 with n = 1: x <- x + (K1 + 2 K2 + 2 K3 + K4) / 6, psi wrapped to (-pi, pi] (time is advanced by
// the caller).  `t` enters with sin/cos of the current attitude (already computed for the controllers).  The four
// stages run as a rolled loop (one copy of the ODE + trig code instead of four: the fully unrolled kernel was
// 128 KB of SASS and stalled on instruction fetch); weights (1,2,2,1) and stage offsets (1/2,1/2,1) are selected by
// the stage index, and acc starts at 0 so acc + 1*K1 == K1 exactly -- the summation order of the reference is kept.
template <typename T, bool ATT_ONLY>
__device__ __forceinline__ void uav_rk44(const Consts<T> &c, T *x, Trig<T> t, T throttle, const T *tq, const T *dis) {
    constexpr int LO = ATT_ONLY ? 6 : 0;
    const T h = c.dt;
    T acc[12], xs[12];
#pragma unroll
    for (int i = LO; i < 12; ++i) { acc[i] = (T)0; xs[i] = x[i]; }
#pragma unroll 1
    for (int s = 0; s < 4; ++s) {
        T d[12];
        uav_ode<T, ATT_ONLY>(c, xs, t, throttle, tq, dis, d);
        const T w = (s == 0 || s == 3) ? (T)1 : (T)2;
        const T cs = (s == 2) ? (T)1 : (T)0.5;
#pragma unroll
        for (int i = LO; i < 12; ++i) {
            const T k = h * d[i];
            acc[i] = acc[i] + w * k;
            xs[i] = x[i] + k * cs;
        }
        if (s < 3) t.eval(xs[6], xs[7], xs[8], !ATT_ONLY);
    }
#pragma unroll
    for (int i = LO; i < 12; ++i) x[i] = x[i] + UAV_DIV(acc[i], (T)6, (T)(1.0 / 6.0));
    if (x[8] > (T)M_PI) x[8] -= (T)(2 * M_PI);
    if (x[8] < (T)-M_PI) x[8] += (T)(2 * M_PI);
}

// FNTSMC sliding surface pieces shared by both loops (FNTSMC.py:61-66 / 128-134), one axis.
template <typename T>
__device__ __forceinline__ void smc_axis(T e, T de, T k1, T gamma, T alpha, T beta, T lmd, T dt, T &integ,
                                         T &s_out, T &dot_s1, T &pa1_de) {
    // |e|^(alpha-1) = exp((alpha-1) log|e|) and |e|^alpha = |e|^(alpha-1) * |e|: one log, one exp and one product for the
    // two powers of FNTSMC.py:61-63 (numpy evaluates two pow()).  e = 0: 0^alpha = 0 (alpha > 0) while 0^(alpha-1) = inf.
    const T ae = Mth<T>::abs(e);
#ifdef B200_STRICT_POW
    // FNTSMC.py:61-66 / 128-134 literally: np.fabs(e) ** alpha, np.fabs(e) ** (alpha - 1), np.fabs(s) ** beta
    const T s_ = de + k1 * e + gamma * Mth<T>::pow(ae, alpha) * Mth<T>::tanh((T)5 * e);
    dot_s1 = Mth<T>::pow(Mth<T>::abs(s_), beta) * Mth<T>::tanh((T)5 * s_);
    integ += dot_s1 * dt;
    s_out = s_ + lmd * integ;
    pa1_de = gamma * alpha * Mth<T>::pow(ae, alpha - (T)1) * de;
    return;
#endif
    const T L = Mth<T>::log_nonneg(ae);
    const T pa1 = pow_from_log<T>(L, alpha - (T)1);
    const T pa_ = pa1 * ae;
    const T pa = alpha == (T)0 ? (T)1 : ((ae == (T)0 && alpha > (T)0) ? (T)0 : pa_);
    const T s = de + k1 * e + gamma * pa * Mth<T>::tanh((T)5 * e);
    dot_s1 = pow_from_log<T>(Mth<T>::log_nonneg(Mth<T>::abs(s)), beta) * Mth<T>::tanh((T)5 * s);
    integ += dot_s1 * dt;
    s_out = s + lmd * integ;           // sigma (att) / so (pos)
    pa1_de = gamma * alpha * pa1 * de; // gamma * alpha * |e|^(alpha-1) * de
}

// -inv(B) . v with B = f1 . diag(1/J) (uav.py:359-360) and inv = LAPACK dgesv(B, I) semantics: LU with partial
// pivoting, then forward/back substitution per unit column, then the 3x3 . 3 product (FNTSMC.py:137).
// Column 0 of B is (1/J0, 0, 0): its multipliers are exactly 0, so only rows 1,2 can be swapped.
template <typename T>
__device__ __forceinline__ void neg_inv_apply(T b00, T b01, T b02, T b11, T b12, T b21, T b22, const T *v, T *out) {
    const bool swap = Mth<T>::abs(b21) > Mth<T>::abs(b11);
    const T u11 = swap ? b21 : b11, u12 = swap ? b22 : b12;
    const T r21 = swap ? b11 : b21, r22 = swap ? b12 : b22;
    const T l = r21 * ((T)1 / u11);
    const T u22 = r22 - l * u12;
    T inv[3][3];
#pragma unroll
    for (int cidx = 0; cidx < 3; ++cidx) {
        // P e_c: rows 1 and 2 exchanged when swap
        T y0 = cidx == 0 ? (T)1 : (T)0;
        T y1 = (cidx == (swap ? 2 : 1)) ? (T)1 : (T)0;
        T y2 = (cidx == (swap ? 1 : 2)) ? (T)1 : (T)0;
        y2 = y2 - l * y1;
        const T x2 = y2 / u22;
        const T x1 = (y1 - u12 * x2) / u11;
        const T x0 = ((y0 - b01 * x1) - b02 * x2) / b00;
        inv[0][cidx] = x0; inv[1][cidx] = x1; inv[2][cidx] = x2;
    }
#pragma unroll
    for (int i = 0; i < 3; ++i) out[i] = -(inv[i][0] * v[0] + inv[i][1] * v[1] + inv[i][2] * v[2]);
}

// Attitude loop: uav_att_ctrl.py:91-108 / uav_pos_ctrl.py:317-337 + FNTSMC.py:112-137 (dd_ref = 0).
// x: full state, t: trig of the current attitude.  Returns torque; also d1 = f1 . pqr (Euler rates).
template <typename T>
__device__ __forceinline__ void att_control(const Consts<T> &c, const T *x, const Trig<T> &t, const T *k1, const T *k2,
                                            const T *gamma, const T *lmd, const T *alpha, const T *beta, T *s1,
                                            const T *ref, const T *dref, T *torque, T *d1) {
    const T p = x[9], q = x[10], r = x[11];
    const T f01 = t.sphi * t.tth, f02 = t.cphi * t.tth, f11 = t.cphi, f12 = -t.sphi;
    const T f21 = UAV_DIV(t.sphi, t.cth, t.rcth), f22 = UAV_DIV(t.cphi, t.cth, t.rcth);
    d1[0] = p + f01 * q + f02 * r;
    d1[1] = f11 * q + f12 * r;
    d1[2] = f21 * q + f22 * r;
    // F() (uav.py:340-354) . rho2
    const T rc2 = t.rcth * t.rcth;
    const T c2 = t.cth * t.cth; // np.cos(theta) ** 2
    (void)c2;
    const T F01 = d1[0] * t.tth * t.cphi + UAV_DIV(d1[1] * t.sphi, c2, rc2);
    const T F02 = -d1[0] * t.tth * t.sphi + UAV_DIV(d1[1] * t.cphi, c2, rc2);
    const T F11 = -d1[0] * t.sphi, F12 = -d1[0] * t.cphi;
    const T F21 = UAV_DIV(d1[0] * t.cphi * t.cth + d1[1] * t.sphi * t.sth, c2, rc2);
    const T F22 = UAV_DIV(-d1[0] * t.sphi * t.cth + d1[1] * t.cphi * t.sth, c2, rc2);
    // f2() (uav.py:302-313)
    const T g0 = UAV_DIV(c.kr * p + q * r * (c.J1 - c.J2), c.J0, c.rJ0);
    const T g1 = UAV_DIV(c.kr * q + p * r * (c.J2 - c.J0), c.J1, c.rJ1);
    const T g2 = UAV_DIV(c.kr * r + p * q * (c.J0 - c.J1), c.J2, c.rJ2);
    T sec[3];
    sec[0] = (F01 * q + F02 * r) + (g0 + f01 * g1 + f02 * g2);
    sec[1] = (F11 * q + F12 * r) + (f11 * g1 + f12 * g2);
    sec[2] = (F21 * q + F22 * r) + (f21 * g1 + f22 * g2);
    T v[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        const T e = x[6 + i] - ref[i], de = d1[i] - dref[i];
        T sigma, dot_s1, pa1_de;
        smc_axis<T>(e, de, k1[i], gamma[i], alpha[i], beta[i], lmd[i], c.dt, s1[i], sigma, dot_s1, pa1_de);
        const T u1 = sec[i] + k1[i] * de + pa1_de + lmd[i] * dot_s1;
        const T u2 = -k2[i] * Mth<T>::tanh((T)10 * sigma);
        v[i] = u1 + u2;
    }
#ifdef B200_UAV_LAPACK_INV
    neg_inv_apply<T>(c.rJ0, f01 * c.rJ1, f02 * c.rJ2, f11 * c.rJ1, f12 * c.rJ2, f21 * c.rJ1, f22 * c.rJ2, v, torque);
#else
    // B = f1 . diag(1/J)  =>  B^-1 = diag(J) . f1^-1 with the closed form
    //   f1^-1 = [[1, 0, -sin th], [0, cos phi, sin phi cos th], [0, -sin phi, cos phi cos th]].
    // The reference calls np.linalg.inv (LU, FNTSMC.py:137); the closed form differs from it only by LAPACK's own
    // rounding (cond(f1) * eps) -- measured in tests/parity_report.py, incl. the near-singular fixtures.
    torque[0] = -c.J0 * (v[0] - t.sth * v[2]);
    torque[1] = -c.J1 * (t.cphi * v[1] + t.sphi * t.cth * v[2]);
    torque[2] = -c.J2 * (t.cphi * t.cth * v[2] - t.sphi * v[1]);
#endif
}


// cos(phi_d) in uo_2_ref_angle_throttle (uav_pos_ctrl.py:339-357 / UavRobust uav_pos_ctrl.py:67-76): the reference
// divides by cos(arcsin(u)).  When u saturates at +-1 that is cos(fl(pi/2)) = +6.1e-17 in fp64 -- theta_d becomes
// +-pi/2 with the sign of the numerator -- but cosf(fl32(pi/2)) = -4.4e-8 < 0 in fp32, which would mirror theta_d
// (measured: 1 % of the steps of the UavHover fixture under U(+-8) actions).  The fp64 path keeps the reference's
// expression bit for bit; the fp32 path uses the identity cos(asin u) = sqrt(1 - u^2) >= 0, which has the fp64 sign.
template <typename T>
__device__ __forceinline__ T cos_of_asin(T u, T phi_d) {
    if (sizeof(T) == 4) return Mth<T>::sqrt(Mth<T>::max(Mth<T>::fma(-u, u, (T)1), (T)0));
    T sn, cs;
    Mth<T>::sincos(phi_d, &sn, &cs); // constant-bank kernels instead of libdevice's cos()
    return cs;
}

// NCH channels of ref_uav / ref_inner at once (ref_cmd.py:4-43).  The training scripts draw ONE period for all channels
// of a trajectory and use the phases (pi/2, 0, 0, 0) (uav_pos_ctrl.py:404-408, train.py:61-66), so channels 1..3 have
// the same angular frequency and the same sincos argument as their predecessor: a channel whose (period, phase) equal
// the previous channel's reuses its w, sin and cos -- the same inputs through the same code give the same bits, so this
// is not an approximation -- and only distinct channels pay for the quotient and the sincos (two instead of four per
// step in the bench configuration).  The test is per thread; lanes with distinct channels simply take the full path.
template <typename T, int NCH>
__device__ __forceinline__ void ref_channels(T time, const T *A, const T *period, const T *bias, const T *phase, T *r,
                                             T *dr, T *ddr) {
    T w = (T)0, s = (T)0, co = (T)1;
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
        if (k == 0 || period[k] != period[k - 1] || phase[k] != phase[k - 1]) {
            // <= 1 ulp from the IEEE quotient (fastmath64.cuh), ~half the instructions
            if (k == 0 || period[k] != period[k - 1]) w = Mth<T>::div((T)(2 * M_PI), period[k]);
            Mth<T>::sincos(w * time + phase[k], &s, &co);
        }
        r[k] = A[k] * s + bias[k];
        dr[k] = A[k] * w * co;
        ddr[k] = -A[k] * (w * w) * s;
    }
}


} // namespace uavk
