// uav.cu -- K-UAVA / K-UAVP: batched UavFntsmcParam attitude and position tracking steps (sm_100a).
//
// One thread = one quadrotor.  A launch performs, for every instance, the whole loop body of the reference's
// train.py: get_param_from_actor(a) -> [ref_uav -> pos FNTSMC -> throttle/angle mapping ->] ref -> attitude FNTSMC
// -> step_update (RK4 of the 12-state ODE, terminal flag, observation, reward) and, optionally, the auto-reset.
//   quadrotor ODE / RK4 / zones      environment/UavFntsmcParam/uav.py:93-148,182-219
//   attitude kinematics f1,f2,F,h    uav.py:285-360
//   controllers                      FNTSMC.py:47-69 (pos), 112-137 (att, with np.linalg.inv)
//   references                       ref_cmd.py:4-43
//   wrappers                         uav_att_ctrl.py:91-128, uav_att_ctrl_RL.py:59-156,
//                                    uav_pos_ctrl.py:302-376,467-486, uav_pos_ctrl_RL.py:59-173
//
// Register-resident design: the 12 ODE states, the RK4 accumulators, both sliding-mode integrators and the gains
// stay in registers for the whole step; sin/cos of (phi, theta, psi) are evaluated once per RK stage and the
// stage-1 values are shared with the controllers (the reference evaluates f1() four times and sin/cos ~60 times).
// HBM traffic is one coalesced read and one coalesced write of each SoA field.
#include "common.cuh"
#ifndef UAV_POS_MINBLOCKS
#define UAV_POS_MINBLOCKS 4
#endif
#ifndef UAV_ATT_MINBLOCKS
#define UAV_ATT_MINBLOCKS 5 // 102 registers: +2.4 % over 4 blocks for the attitude kernel (A/B, end of round 1)
#endif
#include "uav_common.cuh"

namespace {
using namespace uavk;

// uav.py:182-219: 2 position out, 3 attitude out, 1 time out -- evaluated in this order, the last true wins
template <typename T>
__device__ __forceinline__ int terminal_flag(const P &p, const T *x, double time) {
    int flag = 0;
    bool out = false;
#pragma unroll
    for (int i = 0; i < 3; ++i) out = out || (x[i] < (T)p.pos_lo[i]) || (x[i] > (T)p.pos_hi[i]);
    if (out) flag = 2;
    out = false;
#pragma unroll
    for (int i = 0; i < 3; ++i) out = out || (x[6 + i] < (T)p.att_lo[i]) || (x[6 + i] > (T)p.att_hi[i]);
    if (out) flag = 3;
    if (time > p.t_term) flag = 1;
    return flag;
}

// ------------------------------------------------------------------------------------------ attitude env
enum { A_S1 = 6, A_K1 = 9, A_K2 = 12, A_GAM = 15, A_LMD = 18, A_AMP = 21, A_PER = 24, A_PHS = 27, A_REF = 30, A_DREF = 33 };

template <typename T, typename I>
__device__ __forceinline__ void att_reset_state(const P &p, const b200env_io &io, I n, I i, uint64_t seed,
                                               int64_t off, T *x /* out: 12 states */) {
    const uint32_t ep = io.episode[i];
#pragma unroll
    for (int k = 0; k < 6; ++k) { x[k] = (T)0; x[6 + k] = (T)p.init_state[6 + k]; UAV_STS(io.state, n, k, i, x[6 + k]); }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        UAV_STS(io.state, n, A_S1 + k, i, (T)0);
        UAV_STS(io.state, n, A_K1 + k, i, (T)p.att_k1[k]);
        UAV_STS(io.state, n, A_K2 + k, i, (T)p.att_k2[k]);
        UAV_STS(io.state, n, A_GAM + k, i, (T)p.att_gamma[k]);
        UAV_STS(io.state, n, A_LMD + k, i, (T)p.att_lmd[k]);
    }
    double A[3], Tp[3], ph[3];
    if (p.random_trajectory) { // uav_att_ctrl.py:156-161
        Philox rng(seed, (uint64_t)(off + (int64_t)i), ep);
#pragma unroll
        for (int k = 0; k < 3; ++k) A[k] = rng.uniform(0., p.traj_A_hi[k]);
#pragma unroll
        for (int k = 0; k < 3; ++k) Tp[k] = rng.uniform(p.traj_T_lo, p.traj_T_hi);
#pragma unroll
        for (int k = 0; k < 3; ++k) ph[k] = rng.uniform(0., p.traj_phase_hi);
    } else {
#pragma unroll
        for (int k = 0; k < 3; ++k) { A[k] = p.ref_amplitude[k]; Tp[k] = p.ref_period[k]; ph[k] = p.ref_bias_phase[k]; }
    }
    if (p.yaw_fixed) { A[2] = 0.; ph[2] = 0.; }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        UAV_STS(io.state, n, A_AMP + k, i, (T)A[k]);
        UAV_STS(io.state, n, A_PER + k, i, (T)Tp[k]);
        UAV_STS(io.state, n, A_PHS + k, i, (T)ph[k]);
    }
    io.time[i] = 0.0;
    io.episode[i] = ep + 1u;
}

// uav_att_ctrl_RL.py:59-68 (use_norm = False)
template <typename T>
__device__ __forceinline__ void att_observe(const T *x, const Trig<T> &t, const T *ref, const T *dref, T *o) {
    const T q = x[10], r = x[11];
    o[0] = x[6] - ref[0]; o[1] = x[7] - ref[1]; o[2] = x[8] - ref[2];
    o[3] = (x[9] + (t.sphi * t.tth) * q + (t.cphi * t.tth) * r) - dref[0];
    o[4] = (t.cphi * q - t.sphi * r) - dref[1];
    o[5] = ((t.sphi / t.cth) * q + (t.cphi / t.cth) * r) - dref[2];
}

template <typename T, typename I, bool IO32>
__global__ void __launch_bounds__(B200_BLOCK, UAV_ATT_MINBLOCKS)
uav_att_step_kernel(const __grid_constant__ P p, const __grid_constant__ UavDerived dv,
                    const __grid_constant__ b200env_io io, int64_t n_, uint32_t flags, uint64_t seed, int64_t off) {
    const int64_t gi = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gi >= n_) return;
    const I n = (I)n_, i = (I)gi;
    const Consts<T> c(p.m, p.g, p.J, p.kr, p.kt, p.dt, dv);
    T x[12];
#pragma unroll
    for (int k = 0; k < 6; ++k) { x[k] = (T)0; x[6 + k] = UAV_LDS(io.state, n, k, i); }
    double time = io.time[i];
    T s1[3], k1[3], k2[3], gam[3], lmd[3], alpha[3], beta[3], ref[3], dref[3];
    T a[8], rA[3], rT[3], rP[3];
#pragma unroll
    for (int k = 0; k < 8; ++k) a[k] = ldio<T, IO32>(io.action, n, k, i);
    // all loads before the first store (see uav_pos_step_kernel)
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        s1[k] = UAV_LDS(io.state, n, A_S1 + k, i);
        rA[k] = UAV_LDS(io.state, n, A_AMP + k, i); rT[k] = UAV_LDS(io.state, n, A_PER + k, i); rP[k] = UAV_LDS(io.state, n, A_PHS + k, i);
    }
    // get_param_from_actor, uav_att_ctrl_RL.py:141-156: a gain is overwritten only where the actor output is > 0 (N6)
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        k1[k] = a[k] > (T)0 ? (T)10 * a[k] : UAV_LDS(io.state, n, A_K1 + k, i);
        // a / 10 as q = a r, q + (a - 10 q) r with r = RN(1 / 10): the correctly rounded quotient (Markstein; checked
        // against 300 k IEEE quotients incl. float32-valued a), without the IEEE division's slow-path branch
#ifdef B200_STRICT_DIV
        k2[k] = a[k + 3] > (T)0 ? a[k + 3] / (T)10 : UAV_LDS(io.state, n, A_K2 + k, i);
#else
        k2[k] = a[k + 3] > (T)0 ? Divisor<T>((T)10, (T)0.1).div(a[k + 3]) : UAV_LDS(io.state, n, A_K2 + k, i);
#endif
        gam[k] = a[6] > (T)0 ? a[6] : UAV_LDS(io.state, n, A_GAM + k, i);
        lmd[k] = a[7] > (T)0 ? a[7] : UAV_LDS(io.state, n, A_LMD + k, i);
        alpha[k] = (T)p.att_alpha[k];
        beta[k] = (T)p.att_beta[k];
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) { // early write-back
        UAV_STS(io.state, n, A_K1 + k, i, k1[k]);
        UAV_STS(io.state, n, A_K2 + k, i, k2[k]);
        UAV_STS(io.state, n, A_GAM + k, i, gam[k]);
        UAV_STS(io.state, n, A_LMD + k, i, lmd[k]);
    }
    // ref_inner(time, A, T, 0, phase), ref_cmd.py:4-22
    {
        const T zero3[3] = {(T)0, (T)0, (T)0};
        T dd[3];
        ref_channels<T, 3>((T)time, rA, rT, zero3, rP, ref, dref, dd);
    }
    Trig<T> t1;
    t1.eval(x[6], x[7], x[8], false);
    T torque[3], d1[3];
    att_control<T>(c, x, t1, k1, k2, gam, lmd, alpha, beta, s1, ref, dref, torque, d1);
#pragma unroll
    for (int k = 0; k < 3; ++k) UAV_STS(io.state, n, A_S1 + k, i, s1[k]);
    const T u_acc = -(torque[0] * torque[0] * (T)p.R[0] + torque[1] * torque[1] * (T)p.R[1] + torque[2] * torque[2] * (T)p.R[2]);
    if (io.obs) { // current_state = get_state()
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            stio<T, IO32>(io.obs, n, k, i, x[6 + k] - ref[k]);
            stio<T, IO32>(io.obs, n, 3 + k, i, d1[k] - dref[k]);
        }
    }
    // update(): throttle only drives the (zeroed) translational states in att_only mode, uav_att_ctrl.py:110-128
    const T zero3[3] = {(T)0, (T)0, (T)0};
    uav_rk44<T, true>(c, x, t1, (T)0, torque, zero3);
    time += p.dt;
    const int flag = terminal_flag<T>(p, x, time);
    const bool done = (flag == 1) || (flag == 3); // uav_att_ctrl_RL.py:118-127
    Trig<T> t2;
    t2.eval(x[6], x[7], x[8], false);
    T nxt[6];
    att_observe<T>(x, t2, ref, dref, nxt);
    // get_reward, uav_att_ctrl_RL.py:70-106
    const T u_att = -(nxt[0] * nxt[0] * (T)p.Q_e[0] + nxt[1] * nxt[1] * (T)p.Q_e[1] + nxt[2] * nxt[2] * (T)p.Q_e[2]);
    const T u_pqr = -(nxt[3] * nxt[3] * (T)p.Q_de[0] + nxt[4] * nxt[4] * (T)p.Q_de[1] + nxt[5] * nxt[5] * (T)p.Q_de[2]);
    T u_extra = (T)0;
    if (flag == 3) {
        const T nn = (T)((p.time_max - time) / p.dt);
        const T pi2 = (T)(M_PI * M_PI);
        T u_phi = (T)0, u_theta = (T)0;
        if (x[6] > (T)p.att_zone_max[0] || x[6] < (T)p.att_zone_min[0]) u_phi = -pi2 * (T)p.Q_e[0];
        if (x[7] > (T)p.att_zone_max[1] || x[7] < (T)p.att_zone_min[1]) u_theta = -pi2 * (T)p.Q_e[1];
        if (x[8] > (T)p.att_zone_max[2] || x[8] < (T)p.att_zone_min[2]) u_theta = (T)-4 * pi2 * (T)p.Q_e[2]; // sic (N7)
        u_extra = nn * (u_phi + u_theta + u_pqr + u_acc);
    }
    const T reward = u_att + u_pqr + u_acc + u_extra;
#pragma unroll
    for (int k = 0; k < 6; ++k) stio<T, IO32>(io.next_obs, n, k, i, nxt[k]);
    stio<T, IO32>(io.reward, n, 0, i, reward);
    io.done[i] = done ? 1 : 0;
    io.flag[i] = flag;
    if (done && (flags & B200ENV_AUTO_RESET)) {
        T xr[12];
        att_reset_state<T, I>(p, io, n, i, seed, off, xr);
        Trig<T> tr;
        tr.eval(xr[6], xr[7], xr[8], false);
        att_observe<T>(xr, tr, ref, dref, nxt); // first obs of the next episode against the stale ref (reference quirk)
    } else {
#pragma unroll
        for (int k = 0; k < 6; ++k) UAV_STS(io.state, n, k, i, x[6 + k]);
        io.time[i] = time;
        if (done) { // keep the last reference for a later explicit reset()/observe()
#pragma unroll
            for (int k = 0; k < 3; ++k) { UAV_STS(io.state, n, A_REF + k, i, ref[k]); UAV_STS(io.state, n, A_DREF + k, i, dref[k]); }
        }
    }
    if (io.reset_obs) {
#pragma unroll
        for (int k = 0; k < 6; ++k) stio<T, IO32>(io.reset_obs, n, k, i, nxt[k]);
    }
}

template <typename T, bool IO32>
__global__ void __launch_bounds__(B200_BLOCK)
uav_att_reset_kernel(const __grid_constant__ P p, const __grid_constant__ b200env_io io, int64_t n,
                     const uint8_t *mask, uint64_t seed, int64_t off, int observe_only) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (!observe_only && mask && !mask[i]) return;
    T x[12];
    if (observe_only) {
#pragma unroll
        for (int k = 0; k < 6; ++k) { x[k] = (T)0; x[6 + k] = UAV_LDS(io.state, n, k, i); }
    } else {
        att_reset_state<T, int64_t>(p, io, n, i, seed, off, x);
    }
    if (io.next_obs) {
        T ref[3], dref[3], o[6];
#pragma unroll
        for (int k = 0; k < 3; ++k) { ref[k] = UAV_LDS(io.state, n, A_REF + k, i); dref[k] = UAV_LDS(io.state, n, A_DREF + k, i); }
        Trig<T> t;
        t.eval(x[6], x[7], x[8], false);
        att_observe<T>(x, t, ref, dref, o);
#pragma unroll
        for (int k = 0; k < 6; ++k) stio<T, IO32>(io.next_obs, n, k, i, o[k]);
    }
}

// ------------------------------------------------------------------------------------------ position env
enum { P_SIG = 12, P_S1 = 15, P_AREF = 18, P_K1 = 21, P_K2 = 24, P_GAM = 27, P_LMD = 30, P_AMP = 33, P_PER = 37,
       P_PHS = 41, P_PREF = 45, P_DPREF = 48, P_NEXT_PQR0 = 51 /* layout variant 1 only */ };

template <typename T, typename I>
__device__ __forceinline__ void pos_reset_state(const P &p, const b200env_io &io, I n, I i, uint64_t seed,
                                               int64_t off, T *x) {
    const uint32_t ep = io.episode[i];
#pragma unroll
    for (int k = 0; k < 12; ++k) { x[k] = (T)p.init_state[k]; UAV_STS(io.state, n, k, i, x[k]); }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        UAV_STS(io.state, n, P_SIG + k, i, (T)0);
        UAV_STS(io.state, n, P_S1 + k, i, (T)0);
        UAV_STS(io.state, n, P_K1 + k, i, (T)p.pos_k1[k]);
        UAV_STS(io.state, n, P_K2 + k, i, (T)p.pos_k2[k]);
        UAV_STS(io.state, n, P_GAM + k, i, (T)p.pos_gamma[k]);
        UAV_STS(io.state, n, P_LMD + k, i, (T)p.pos_lmd[k]);
    }
    double A[4], Tp[4], ph[4];
    Philox rng(seed, (uint64_t)(off + (int64_t)i), ep);
    if (p.random_trajectory) { // uav_pos_ctrl.py:404-408
        const double a = rng.uniform(0., p.traj_A_hi[0]);
        const double tt = rng.uniform(p.traj_T_lo, p.traj_T_hi);
        A[0] = A[1] = A[2] = a; A[3] = 0.;
#pragma unroll
        for (int k = 0; k < 4; ++k) { Tp[k] = tt; ph[k] = p.ref_bias_phase[k]; }
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) { A[k] = p.ref_amplitude[k]; Tp[k] = p.ref_period[k]; ph[k] = p.ref_bias_phase[k]; }
    }
    if (p.yaw_fixed) { A[3] = 0.; ph[3] = 0.; }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        UAV_STS(io.state, n, P_AMP + k, i, (T)A[k]);
        UAV_STS(io.state, n, P_PER + k, i, (T)Tp[k]);
        UAV_STS(io.state, n, P_PHS + k, i, (T)ph[k]);
    }
    if (p.random_pos0) { // uav_pos_ctrl.py:510-513 -> set_random_init_pos :457-465 -> reset_uav_with_param uav.py:252-268
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            // trajectory[0][k] = bias_a + A sin(2 pi / T * 0 + phase)                       uav_pos_ctrl.py:386-390
            const double t0 = p.ref_bias_a[k] + A[k] * ::sin(ph[k]);
            const double r = ::fabs(p.init_pos_r[k]);
            const double pos0 = rng.uniform(t0 - r, t0 + r);
            x[k] = (T)pos0;
            x[9 + k] = UAV_LDS(io.state, n, P_NEXT_PQR0 + k, i); // new_param.pqr0 = init_state[9:12] = the previous pos0 (N5)
            UAV_STS(io.state, n, k, i, x[k]);
            UAV_STS(io.state, n, 9 + k, i, x[9 + k]);
            UAV_STS(io.state, n, P_NEXT_PQR0 + k, i, x[k]);      // init_state = concat(pos0, vel0, angle0, pos0)
        }
    }
    // att_ref is not reset by the reference (uav_pos_ctrl.py:488-533): left as stored
    io.time[i] = 0.0;
    io.episode[i] = ep + 1u;
}

// one instance, one control period (the body of the step kernel)
template <typename T, typename I, bool IO32>
__device__ __forceinline__ void uav_pos_step_one(const P &p, const Consts<T> &c, const b200env_io &io, I n, I i,
                                                 uint32_t flags, uint64_t seed, int64_t off) {
    T x[12];
#pragma unroll
    for (int k = 0; k < 12; ++k) x[k] = UAV_LDS(io.state, n, k, i);
    double time = io.time[i];
    T a[8], dis[3] = {(T)0, (T)0, (T)0};
#pragma unroll
    for (int k = 0; k < 8; ++k) a[k] = ldio<T, IO32>(io.action, n, k, i);
    if (io.dis) {
#pragma unroll
        for (int k = 0; k < 3; ++k) dis[k] = ldio<T, IO32>(io.dis, n, k, i);
    }
    // All loads are issued here, before the first store: the compiler cannot move a load above a store to the same
    // buffer (possible aliasing), and a mid-kernel DRAM load is not hidden by the 4 resident warps per scheduler.
    T sig[3], s1[3], aref0, aref1, rA[4], rT[4], rP[4];
#pragma unroll
    for (int k = 0; k < 3; ++k) { sig[k] = UAV_LDS(io.state, n, P_SIG + k, i); s1[k] = UAV_LDS(io.state, n, P_S1 + k, i); }
    aref0 = UAV_LDS(io.state, n, P_AREF + 0, i);
    aref1 = UAV_LDS(io.state, n, P_AREF + 1, i);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        rA[k] = UAV_LDS(io.state, n, P_AMP + k, i); rT[k] = UAV_LDS(io.state, n, P_PER + k, i); rP[k] = UAV_LDS(io.state, n, P_PHS + k, i);
    }
    // Every persistent field is written back as soon as its new value is known (short register live ranges; a later
    // auto-reset simply overwrites what it redefines).
    // ---- get_param_from_actor, uav_pos_ctrl_RL.py:158-173: a gain changes only where the actor output is > 0 (N6)
    T k1[3], k2[3], gam[3], lmd[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        k1[k] = a[k] > (T)0 ? a[k] : UAV_LDS(io.state, n, P_K1 + k, i);
        k2[k] = a[k + 3] > (T)0 ? a[k + 3] : UAV_LDS(io.state, n, P_K2 + k, i);
        gam[k] = a[6] > (T)0 ? a[6] : UAV_LDS(io.state, n, P_GAM + k, i);
        lmd[k] = a[7] > (T)0 ? a[7] : UAV_LDS(io.state, n, P_LMD + k, i);
        UAV_STS(io.state, n, P_K1 + k, i, k1[k]);
        UAV_STS(io.state, n, P_K2 + k, i, k2[k]);
        UAV_STS(io.state, n, P_GAM + k, i, gam[k]);
        UAV_STS(io.state, n, P_LMD + k, i, lmd[k]);
    }
    // ---- ref_uav(time, A, T, bias, phase), ref_cmd.py:25-43
    T ref[4], dref[4], ddref[4];
    {
        const T bias4[4] = {(T)p.ref_bias_a[0], (T)p.ref_bias_a[1], (T)p.ref_bias_a[2], (T)p.ref_bias_a[3]};
        ref_channels<T, 4>((T)time, rA, rT, bias4, rP, ref, dref, ddref);
    }
    // ---- pos_control, uav_pos_ctrl.py:302-315 + FNTSMC.py:47-69 (obs = 0)
    T ctrl[3];
    const T kt_m = c.kt_m; // kt / m (uav_pos_ctrl.py:310), constant: the compiler folds it from the kernel arguments
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const T e = x[k] - ref[k], de = x[3 + k] - dref[k];
        T so, dso1, pa1_de;
        smc_axis<T>(e, de, k1[k], gam[k], (T)p.pos_alpha[k], (T)p.pos_beta[k], lmd[k], c.dt, sig[k], so, dso1, pa1_de);
        UAV_STS(io.state, n, P_SIG + k, i, sig[k]);
        const T uo1 = kt_m * x[3 + k] + ddref[k] - k1[k] * de - pa1_de - lmd[k] * dso1;
        const T uo2 = -k2[k] * so;
        ctrl[k] = uo1 + uo2;
    }
    const T u_acc = -(ctrl[0] * ctrl[0] * (T)p.R[0] + ctrl[1] * ctrl[1] * (T)p.R[1] + ctrl[2] * ctrl[2] * (T)p.R[2]);
    Trig<T> t1;
    t1.eval(x[6], x[7], x[8], true);
    // ---- uo_2_ref_angle_throttle(limit = pi/4), uav_pos_ctrl.py:339-357
    const T uf = (ctrl[2] + c.g) * c.m / (t1.cphi * t1.cth);
    const T asin_phi_d = clampc<T>(Mth<T>::div((ctrl[0] * t1.spsi - ctrl[1] * t1.cpsi) * c.m, uf), (T)-1, (T)1);
    T phi_d = Mth<T>::asin(asin_phi_d);
    const T asin_theta_d = clampc<T>(
        Mth<T>::div((ctrl[0] * t1.cpsi + ctrl[1] * t1.spsi) * c.m, uf * cos_of_asin<T>(asin_phi_d, phi_d)), (T)-1, (T)1);
    T theta_d = Mth<T>::asin(asin_theta_d);
    const T lim = (T)p.att_limit;
    phi_d = clampc<T>(phi_d, -lim, lim);
    theta_d = clampc<T>(theta_d, -lim, lim);
    // ---- generate_action_4_uav, uav_pos_ctrl.py:470-481: finite-difference reference rates, clipped, integrated back
    T rho_d[3] = {phi_d, theta_d, ref[3]};
#ifdef B200_STRICT_DIV
    T drho_d[3] = {(phi_d - aref0) / c.dt, (theta_d - aref1) / c.dt, dref[3]};
#else
    const Divisor<T> by_dt(c.dt);
    T drho_d[3] = {by_dt.div(phi_d - aref0), by_dt.div(theta_d - aref1), dref[3]};
#endif
    const T rl = (T)p.dot_att_ref_limit;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        drho_d[k] = clampc<T>(drho_d[k], -rl, rl);
        rho_d[k] = rho_d[k] + drho_d[k] * c.dt;
        UAV_STS(io.state, n, P_AREF + k, i, rho_d[k]); // att_ref = rho_d (persists across resets, uav_pos_ctrl.py:329)
    }
    // ---- att_control, uav_pos_ctrl.py:317-337
    T torque[3], d1[3], ak1[3], ak2[3], agam[3], almd[3], aalpha[3], abeta[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        ak1[k] = (T)p.att_k1[k]; ak2[k] = (T)p.att_k2[k]; agam[k] = (T)p.att_gamma[k]; almd[k] = (T)p.att_lmd[k];
        aalpha[k] = (T)p.att_alpha[k]; abeta[k] = (T)p.att_beta[k];
    }
    att_control<T>(c, x, t1, ak1, ak2, agam, almd, aalpha, abeta, s1, rho_d, drho_d, torque, d1);
#pragma unroll
    for (int k = 0; k < 3; ++k) UAV_STS(io.state, n, P_S1 + k, i, s1[k]);
    if (io.obs) { // current_state = get_state(), uav_pos_ctrl_RL.py:59-68
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            stio<T, IO32>(io.obs, n, k, i, x[k] - ref[k]);
            stio<T, IO32>(io.obs, n, 3 + k, i, x[3 + k] - dref[k]);
        }
    }
    // ---- update(): rk44(action, dis, n = 1), uav_pos_ctrl.py:359-376
    uav_rk44<T, false>(c, x, t1, uf, torque, dis);
    time += p.dt;
    const int flag = terminal_flag<T>(p, x, time);
    const bool done = flag != 0; // uav_pos_ctrl_RL.py:132-143
    T nxt[6];
#pragma unroll
    for (int k = 0; k < 3; ++k) { nxt[k] = x[k] - ref[k]; nxt[3 + k] = x[3 + k] - dref[k]; }
    // ---- get_reward, uav_pos_ctrl_RL.py:82-120
    const T u_pos = -(nxt[0] * nxt[0] * (T)p.Q_e[0] + nxt[1] * nxt[1] * (T)p.Q_e[1] + nxt[2] * nxt[2] * (T)p.Q_e[2]);
    const T u_vel = -(nxt[3] * nxt[3] * (T)p.Q_de[0] + nxt[4] * nxt[4] * (T)p.Q_de[1] + nxt[5] * nxt[5] * (T)p.Q_de[2]);
    T u_extra = (T)0;
    if (flag == 2 || flag == 3) {
        const T nn = (T)((p.time_max - time) / p.dt);
        u_extra = nn * (u_pos + u_vel + u_acc);
    }
    const T reward = u_pos + u_vel + u_acc + u_extra;
#pragma unroll
    for (int k = 0; k < 6; ++k) stio<T, IO32>(io.next_obs, n, k, i, nxt[k]);
    stio<T, IO32>(io.reward, n, 0, i, reward);
    io.done[i] = done ? 1 : 0;
    io.flag[i] = flag;
    if (done && (flags & B200ENV_AUTO_RESET)) {
        T xr[12];
        pos_reset_state<T, I>(p, io, n, i, seed, off, xr);
#pragma unroll
        for (int k = 0; k < 3; ++k) { nxt[k] = xr[k] - ref[k]; nxt[3 + k] = xr[3 + k] - dref[k]; } // stale pos_ref (quirk)
    } else {
#pragma unroll
        for (int k = 0; k < 12; ++k) UAV_STS(io.state, n, k, i, x[k]);
        io.time[i] = time;
        if (done) { // keep the last reference for a later explicit reset()/observe()
#pragma unroll
            for (int k = 0; k < 3; ++k) { UAV_STS(io.state, n, P_PREF + k, i, ref[k]); UAV_STS(io.state, n, P_DPREF + k, i, dref[k]); }
        }
    }
    if (io.reset_obs) {
#pragma unroll
        for (int k = 0; k < 6; ++k) stio<T, IO32>(io.reset_obs, n, k, i, nxt[k]);
    }
}

template <typename T, typename I, bool IO32>
__global__ void __launch_bounds__(B200_BLOCK, UAV_POS_MINBLOCKS)
uav_pos_step_kernel(const __grid_constant__ P p, const __grid_constant__ UavDerived dv,
                    const __grid_constant__ b200env_io io, int64_t n_, uint32_t flags, uint64_t seed, int64_t off) {
    const int64_t gi = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gi >= n_) return;
    const Consts<T> c(p.m, p.g, p.J, p.kr, p.kt, p.dt, dv);
    uav_pos_step_one<T, I, IO32>(p, c, io, (I)n_, (I)gi, flags, seed, off);
}

template <typename T, bool IO32>
__global__ void __launch_bounds__(B200_BLOCK)
uav_pos_reset_kernel(const __grid_constant__ P p, const __grid_constant__ b200env_io io, int64_t n,
                     const uint8_t *mask, uint64_t seed, int64_t off, int observe_only) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (!observe_only && mask && !mask[i]) return;
    T x[12];
    if (observe_only) {
#pragma unroll
        for (int k = 0; k < 12; ++k) x[k] = UAV_LDS(io.state, n, k, i);
    } else {
        pos_reset_state<T, int64_t>(p, io, n, i, seed, off, x);
    }
    if (io.next_obs) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            stio<T, IO32>(io.next_obs, n, k, i, x[k] - UAV_LDS(io.state, n, P_PREF + k, i));
            stio<T, IO32>(io.next_obs, n, 3 + k, i, x[3 + k] - UAV_LDS(io.state, n, P_DPREF + k, i));
        }
    }
}

} // namespace

#define UAV_LAUNCH(kern, ...) B200_LAUNCH_TIO(kern, b200_grid(n), B200_BLOCK, s, __VA_ARGS__)

// step kernels: 32-bit SoA index arithmetic whenever every [field][n] offset fits in 32 bits
#define UAV_LAUNCH_STEP(kern, fields, gridexpr, ...)                                                                        \
    do {                                                                                                           \
        const bool i32 = (int64_t)(fields) * n < ((int64_t)1 << 32);                                               \
        const bool o32 = b200_io32(io);                                                                            \
        const unsigned g = (gridexpr);                                                                             \
        if (dtype == B200ENV_F64) {                                                                                \
            if (i32 && o32) kern<double, uint32_t, true><<<g, B200_BLOCK, 0, s>>>(__VA_ARGS__);                    \
            else if (i32) kern<double, uint32_t, false><<<g, B200_BLOCK, 0, s>>>(__VA_ARGS__);                     \
            else if (o32) kern<double, int64_t, true><<<g, B200_BLOCK, 0, s>>>(__VA_ARGS__);                       \
            else kern<double, int64_t, false><<<g, B200_BLOCK, 0, s>>>(__VA_ARGS__);                               \
        } else {                                                                                                   \
            if (i32) kern<float, uint32_t, false><<<g, B200_BLOCK, 0, s>>>(__VA_ARGS__);                           \
            else kern<float, int64_t, false><<<g, B200_BLOCK, 0, s>>>(__VA_ARGS__);                                \
        }                                                                                                          \
    } while (0)

int uav_att_dims(int variant, int *sf, int *od, int *ad, int *dd) {
    if (variant != 0) return B200ENV_EENV;
    if (sf) *sf = B200_UAV_ATT_STATE_FIELDS;
    if (od) *od = 6;
    if (ad) *ad = 8;
    if (dd) *dd = 0;
    return B200ENV_OK;
}
int uav_pos_dims(int variant, int *sf, int *od, int *ad, int *dd) {
    if (variant != 0 && variant != 1) return B200ENV_EENV;
    if (sf) *sf = variant == 1 ? B200_UAV_POS_STATE_FIELDS_V1 : B200_UAV_POS_STATE_FIELDS;
    if (od) *od = 6;
    if (ad) *ad = 8;
    if (dd) *dd = 3;
    return B200ENV_OK;
}

static int uav_check_step(const b200env_io *io, uint32_t flags) {
    if (!io->state || !io->time || !io->action || !io->next_obs || !io->reward || !io->done || !io->flag) return B200ENV_ENULL;
    if ((flags & B200ENV_AUTO_RESET) && !io->episode) return B200ENV_ENULL;
    return B200ENV_OK;
}

int uav_att_step(int dtype, int64_t n, const void *params, const b200env_io *io, uint32_t flags, uint64_t seed,
                 int64_t off, cudaStream_t s) {
    int rc = uav_check_step(io, flags);
    if (rc) return rc;
    const P &p = *static_cast<const P *>(params);
    UAV_LAUNCH_STEP(uav_att_step_kernel, B200_UAV_ATT_STATE_FIELDS, b200_grid(n), p, uav_derive(p.m, p.J, p.kt), *io, n, flags, seed, off);
    return b200_check_launch();
}
int uav_pos_step(int dtype, int64_t n, const void *params, const b200env_io *io, uint32_t flags, uint64_t seed,
                 int64_t off, cudaStream_t s) {
    int rc = uav_check_step(io, flags);
    if (rc) return rc;
    const P &p = *static_cast<const P *>(params);
    UAV_LAUNCH_STEP(uav_pos_step_kernel, B200_UAV_POS_STATE_FIELDS_V1, b200_grid(n), p, uav_derive(p.m, p.J, p.kt), *io, n, flags, seed, off);
    return b200_check_launch();
}
int uav_att_reset(int dtype, int64_t n, const void *params, const b200env_io *io, const uint8_t *mask, uint64_t seed,
                  int64_t off, cudaStream_t s) {
    if (!io->state || !io->time || !io->episode) return B200ENV_ENULL;
    const P &p = *static_cast<const P *>(params);
    UAV_LAUNCH(uav_att_reset_kernel, p, *io, n, mask, seed, off, 0);
    return b200_check_launch();
}
int uav_pos_reset(int dtype, int64_t n, const void *params, const b200env_io *io, const uint8_t *mask, uint64_t seed,
                  int64_t off, cudaStream_t s) {
    if (!io->state || !io->time || !io->episode) return B200ENV_ENULL;
    const P &p = *static_cast<const P *>(params);
    UAV_LAUNCH(uav_pos_reset_kernel, p, *io, n, mask, seed, off, 0);
    return b200_check_launch();
}
int uav_att_observe(int dtype, int64_t n, const void *params, const b200env_io *io, cudaStream_t s) {
    if (!io->state || !io->time || !io->next_obs) return B200ENV_ENULL;
    const P &p = *static_cast<const P *>(params);
    UAV_LAUNCH(uav_att_reset_kernel, p, *io, n, nullptr, 0, 0, 1);
    return b200_check_launch();
}
int uav_pos_observe(int dtype, int64_t n, const void *params, const b200env_io *io, cudaStream_t s) {
    if (!io->state || !io->time || !io->next_obs) return B200ENV_ENULL;
    const P &p = *static_cast<const P *>(params);
    UAV_LAUNCH(uav_pos_reset_kernel, p, *io, n, nullptr, 0, 0, 1);
    return b200_check_launch();
}
