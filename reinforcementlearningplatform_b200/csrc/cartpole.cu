// cartpole.cu -- K-CP: batched CartPole / CartPoleAngleOnly step (sm_100a).
//
// Replaces, for n instances at once,
//   environment/CartPole/CartPole.py:145-295            (variant 0)
//   environment/CartPole/CartPoleAngleOnly.py:139-299   (variant 1)
//   demonstration/PPO2/PPO2-4-CartPoleAngleOnly/cartpole_angleonly.py:137-279 (variant 2)
//
// One thread = one instance; the four ODE states, `time` and the force live in
// registers for the whole control period (10|11 RK4 sub-steps of h = dt/10 for
// variants 0/1 -- the reference's `while self.time < tt` loop on an fp64 time
// accumulated with plain adds, note N1 -- or one step of size dt for variant 2).
#include <type_traits>
#include "common.cuh"

namespace {

template <typename T>
struct CartPole {
    T theta, dtheta, x, dx;
    double time;

    // constants hoisted out of the ODE, grouped as the reference's left-to-right products
    T mell, kf, c34mg, Mm, c34m, c34_m_ell, mg, m, force;

    __device__ __forceinline__ void init_consts(const b200_cartpole_params &p) {
        mell = (T)(p.m * p.ell);               // self.m * self.ell
        kf = (T)p.kf;
        c34mg = (T)(3.0 / 4.0 * p.m * p.g);    // 3 / 4 * self.m * self.g
        Mm = (T)(p.M + p.m);                   // self.M + self.m
        c34m = (T)(3.0 / 4.0 * p.m);           // 3 / 4 * self.m
        c34_m_ell = (T)(3.0 / 4.0 / p.m / p.ell);
        mg = (T)(p.m * p.g);
        m = (T)p.m;
    }

    // CartPole.py:219-238
    __device__ __forceinline__ void ode(T th, T dth, T dxx, T &ddth, T &ddx) const {
        T s, c;
        Mth<T>::sincos(th, &s, &c);
        ddx = (force + mell * (dth * dth) * s - kf * dxx - c34mg * s * c) / (Mm - c34m * (c * c));
        ddth = c34_m_ell * (mg * s - m * ddx * c);
    }

    // one RK4 sub-step of size h, CartPole.py:246-251
    __device__ __forceinline__ void rk4(T h) {
        const T half = (T)0.5;
        T a1, b1, a2, b2, a3, b3, a4, b4;
        ode(theta, dtheta, dx, a1, b1);
        const T k1_th = h * dtheta, k1_dth = h * a1, k1_x = h * dx, k1_dx = h * b1;
        ode(theta + k1_th * half, dtheta + k1_dth * half, dx + k1_dx * half, a2, b2);
        const T k2_th = h * (dtheta + k1_dth * half), k2_dth = h * a2, k2_x = h * (dx + k1_dx * half), k2_dx = h * b2;
        ode(theta + k2_th * half, dtheta + k2_dth * half, dx + k2_dx * half, a3, b3);
        const T k3_th = h * (dtheta + k2_dth * half), k3_dth = h * a3, k3_x = h * (dx + k2_dx * half), k3_dx = h * b3;
        ode(theta + k3_th, dtheta + k3_dth, dx + k3_dx, a4, b4);
        const T k4_th = h * (dtheta + k3_dth), k4_dth = h * a4, k4_x = h * (dx + k3_dx), k4_dx = h * b4;
        const T two = (T)2, six = (T)6;
        theta = theta + div6<T>(k1_th + two * k2_th + two * k3_th + k4_th);
        dtheta = dtheta + div6<T>(k1_dth + two * k2_dth + two * k3_dth + k4_dth);
        x = x + div6<T>(k1_x + two * k2_x + two * k3_x + k4_x);
        dx = dx + div6<T>(k1_dx + two * k2_dx + two * k3_dx + k4_dx);
    }

    // get_state(): CartPole.py:145-153 / cartpole_angleonly.py:137-143
    __device__ __forceinline__ void observe(const b200_cartpole_params &p, T *o) const {
        const T g = (T)p.static_gain;
        const Divisor<T> d0((T)p.theta_max);
        o[0] = d0.div(theta) * g;
        if (p.variant == 0) {
            const Divisor<T> d1((T)p.dtheta_max), d2((T)p.x_max), d3((T)p.dx_max);
            o[1] = d1.div(dtheta) * g;
            o[2] = d2.div(x) * g;
            o[3] = d3.div(dx) * g;
        } else {
            const Divisor<T> d1((T)p.norm_boundless);
            o[1] = d1.div(dtheta) * g;
        }
    }

    __device__ __forceinline__ void reset(const b200_cartpole_params &p, uint64_t seed, uint64_t gid, uint32_t ep) {
        Philox rng(seed, gid, ep);
        const double th0 = rng.uniform(p.reset_theta_lo, p.reset_theta_hi); // CartPole.py:272
        const double x0 = rng.uniform(p.reset_x_lo, p.reset_x_hi);          // CartPole.py:273
        theta = (T)th0;
        x = (T)x0;
        dtheta = (T)0;
        dx = (T)0;
        time = 0.0;
    }
};

template <typename T>
__device__ __forceinline__ void load_state(CartPole<T> &e, const b200env_io &io, int64_t n, int64_t i) {
    e.theta = ld<T>(io.state, n, 0, i);
    e.dtheta = ld<T>(io.state, n, 1, i);
    e.x = ld<T>(io.state, n, 2, i);
    e.dx = ld<T>(io.state, n, 3, i);
    e.time = io.time[i];
}
template <typename T>
__device__ __forceinline__ void store_state(const CartPole<T> &e, const b200env_io &io, int64_t n, int64_t i) {
    st<T>(io.state, n, 0, i, e.theta);
    st<T>(io.state, n, 1, i, e.dtheta);
    st<T>(io.state, n, 2, i, e.x);
    st<T>(io.state, n, 3, i, e.dx);
    io.time[i] = e.time;
}

// Row pointers of one control period: the b200env_io buffers of a single step, or row t of a time-major rollout.
struct StepRows {
    const void *action;
    void *obs, *next_obs, *reward;
    uint8_t *done;
    int32_t *flag;
};

// step_update(action) of one instance whose state is in `e` (registers): current_state, rk44, is_Terminal, next_state,
// get_reward, stores of this step's outputs, auto-reset.  `ep` is the instance's episode counter (register copy).
// On return nxt holds what the policy sees next (next_state, or the reset observation).
template <typename T, bool IO32>
__device__ __forceinline__ void cartpole_step_body(CartPole<T> &e, const b200_cartpole_params &p, const StepRows &r,
                                                   int64_t n, int64_t i, uint32_t flags, uint64_t seed, int64_t off,
                                                   uint32_t &ep, T (&nxt)[4]) {
    const int obs_dim = p.variant == 0 ? 4 : 2;
    e.force = ldio<T, IO32>(r.action, n, 0, i);

    T cur[4];
    e.observe(p, cur); // self.current_state = self.get_state()
    if (r.obs) {
        for (int k = 0; k < obs_dim; ++k) stio<T, IO32>(r.obs, n, k, i, cur[k]);
    }

    // ---- rk44
    if (p.variant == 2) {
        e.rk4((T)p.dt); // cartpole_angleonly.py:218-229
        e.time += p.dt;
    } else {
        const double h = p.dt / 10.0;      // CartPole.py:242
        const double tt = e.time + p.dt;   // CartPole.py:243
        const T hT = (T)h;
        while (e.time < tt) {              // 10 or 11 trips, decided by fp64 rounding of time (N1)
            e.rk4(hT);
            e.time += h;
        }
    }

    // ---- is_Terminal
    int flag = 0;
    bool done = false;
    const bool angle_out = (e.theta > (T)p.theta_term_hi) || (e.theta < (T)p.theta_term_lo);
    if (p.variant == 0) { // CartPole.py:160-185: every test runs, the last true one wins (N3)
        if (angle_out) { flag = 1; done = true; }
        if (e.x > (T)p.x_max || e.x < -(T)p.x_max) { flag = 2; done = true; }
        if (e.time > p.time_max) { flag = 3; done = true; }
        const T ex = (T)0 - e.x, eth = (T)0 - e.theta;
        if (Mth<T>::sqrt(sumsq_rn(ex, e.dx, eth, e.dtheta)) < (T)1e-2) { flag = 4; done = true; } // no FMA: common.cuh
    } else if (p.variant == 1) { // CartPoleAngleOnly.py:144-166: returns at the first true test
        if (angle_out) { flag = 1; done = true; }
        else if (e.time > p.time_max) { flag = 3; done = true; }
    } else { // cartpole_angleonly.py:150-168
        if (angle_out) { flag = 1; done = true; }
        if (e.time > p.time_max) { flag = 3; done = true; }
        const T eth = (T)0 - e.theta;
        if (Mth<T>::sqrt(sumsq_rn(eth, e.dtheta)) < (T)1e-2) { flag = 4; done = true; }
    }

    e.observe(p, nxt);

    // ---- get_reward
    T reward;
    if (p.variant == 0) { // CartPole.py:187-217
        const T r_x = -Mth<T>::abs(e.x) * (T)5;
        const T r_th = -Mth<T>::abs(e.theta) * (T)1;
        const T r_f = -Mth<T>::abs(e.force) * (T)0.01;
        const T sum = r_x + r_th + r_f; // the two zero-weighted terms add -0.0 and do not change the sum
        T extra = (T)0;
        if (flag == 1 || flag == 2) {
            const T nn = (T)((p.time_max - e.time) / p.dt);
            extra = nn * sum;
        }
        reward = sum + extra;
    } else if (p.variant == 1) { // CartPoleAngleOnly.py:188-208
        // rad2deg(s[0] / staticGain * thetaMax) = (...) * 180. / np.pi
        const T ce = Mth<T>::abs(cur[0] / (T)p.static_gain * (T)p.theta_max * (T)180.0 / (T)M_PI);
        const T ne = Mth<T>::abs(nxt[0] / (T)p.static_gain * (T)p.theta_max * (T)180.0 / (T)M_PI);
        T rr = ne > ce ? (T)-2 : (ne == ce ? (T)0 : (T)2);
        if (ce <= (T)0.5 && ne <= (T)0.5) rr += (T)5;
        if (flag == 1) rr -= (T)100;
        else if (flag == 3) rr += (T)500;
        reward = rr;
    } else { // cartpole_angleonly.py:170-195
        const T r1 = -(e.theta * e.theta) * (T)10;
        T r4 = (T)0;
        if (flag == 1) {
            const T nn = (T)((p.time_max - e.time) / p.dt);
            r4 = nn * r1;
        }
        reward = r1 + r4;
    }

    for (int k = 0; k < obs_dim; ++k) stio<T, IO32>(r.next_obs, n, k, i, nxt[k]);
    stio<T, IO32>(r.reward, n, 0, i, reward);
    r.done[i] = done ? 1 : 0;
    r.flag[i] = flag;

    if (done && (flags & B200ENV_AUTO_RESET)) {
        e.reset(p, seed, (uint64_t)(off + i), ep);
        ++ep;
        e.observe(p, nxt);
    }
}

template <typename T, bool IO32>
__global__ void __launch_bounds__(B200_BLOCK)
cartpole_step_kernel(const __grid_constant__ b200_cartpole_params p, const __grid_constant__ b200env_io io,
                     int64_t n, uint32_t flags, uint64_t seed, int64_t off) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    CartPole<T> e;
    e.init_consts(p);
    load_state(e, io, n, i);
    const bool ar = (flags & B200ENV_AUTO_RESET) != 0;
    uint32_t ep = ar ? io.episode[i] : 0u;
    const uint32_t ep0 = ep;
    const StepRows r = {io.action, io.obs, io.next_obs, io.reward, io.done, io.flag};
    T nxt[4];
    cartpole_step_body<T, IO32>(e, p, r, n, i, flags, seed, off, ep, nxt);
    if (ep != ep0) io.episode[i] = ep;
    if (io.reset_obs) {
        const int obs_dim = p.variant == 0 ? 4 : 2;
        for (int k = 0; k < obs_dim; ++k) stio<T, IO32>(io.reset_obs, n, k, i, nxt[k]);
    }
    store_state(e, io, n, i);
}

// b200env_rollout: rs.steps control periods in ONE launch, the four ODE states, time and the episode counter in
// registers from the first step to the last (config #2: 65,536 instances x 1000 steps would otherwise pay 1000 launches
// of a 19 us kernel, each re-reading and re-writing the state).  Row t of every time-major array is `stride` elements
// after row t - 1 (b200env_rollout_spec).
template <typename T, bool IO32>
__global__ void __launch_bounds__(B200_BLOCK)
cartpole_rollout_kernel(const __grid_constant__ b200_cartpole_params p, const __grid_constant__ b200env_io io,
                        const __grid_constant__ b200env_rollout_spec rs, int64_t n, uint32_t flags, uint64_t seed,
                        int64_t off) {
    typedef typename std::conditional<IO32, float, T>::type TIO;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    CartPole<T> e;
    e.init_consts(p);
    load_state(e, io, n, i);
    const bool ar = (flags & B200ENV_AUTO_RESET) != 0;
    uint32_t ep = ar ? io.episode[i] : 0u;
    const uint32_t ep0 = ep;
    T nxt[4] = {};
    for (int64_t t = 0; t < rs.steps; ++t) {
        StepRows r;
        r.action = static_cast<const TIO *>(io.action) + t * rs.action_stride;
        r.obs = io.obs ? static_cast<TIO *>(io.obs) + t * rs.obs_stride : nullptr;
        r.next_obs = static_cast<TIO *>(io.next_obs) + t * rs.next_obs_stride;
        r.reward = static_cast<TIO *>(io.reward) + t * rs.reward_stride;
        r.done = io.done + t * rs.done_stride;
        r.flag = io.flag + t * rs.flag_stride;
        cartpole_step_body<T, IO32>(e, p, r, n, i, flags, seed, off, ep, nxt);
    }
    if (ep != ep0) io.episode[i] = ep;
    if (io.reset_obs) {
        const int obs_dim = p.variant == 0 ? 4 : 2;
        for (int k = 0; k < obs_dim; ++k) stio<T, IO32>(io.reset_obs, n, k, i, nxt[k]);
    }
    store_state(e, io, n, i);
}

template <typename T, bool IO32>
__global__ void __launch_bounds__(B200_BLOCK)
cartpole_reset_kernel(const __grid_constant__ b200_cartpole_params p, const __grid_constant__ b200env_io io,
                      int64_t n, const uint8_t *mask, uint64_t seed, int64_t off, int observe_only) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (!observe_only && mask && !mask[i]) return;
    CartPole<T> e;
    if (observe_only) {
        load_state(e, io, n, i);
    } else {
        const uint32_t ep = io.episode[i];
        e.reset(p, seed, (uint64_t)(off + i), ep);
        io.episode[i] = ep + 1u;
        store_state(e, io, n, i);
    }
    if (io.next_obs) {
        T o[4];
        e.observe(p, o);
        const int obs_dim = p.variant == 0 ? 4 : 2;
        for (int k = 0; k < obs_dim; ++k) stio<T, IO32>(io.next_obs, n, k, i, o[k]);
    }
}

} // namespace

int cartpole_dims(int variant, int *sf, int *od, int *ad, int *dd) {
    if (variant < 0 || variant > 2) return B200ENV_EENV;
    if (sf) *sf = B200_CARTPOLE_STATE_FIELDS;
    if (od) *od = variant == 0 ? 4 : 2;
    if (ad) *ad = 1;
    if (dd) *dd = 0;
    return B200ENV_OK;
}

int cartpole_step(int dtype, int64_t n, const void *params, const b200env_io *io, uint32_t flags,
                  uint64_t seed, int64_t off, cudaStream_t s) {
    const b200_cartpole_params &p = *static_cast<const b200_cartpole_params *>(params);
    if (p.variant < 0 || p.variant > 2) return B200ENV_EENV;
    if (!io->state || !io->time || !io->action || !io->next_obs || !io->reward || !io->done || !io->flag)
        return B200ENV_ENULL;
    if ((flags & B200ENV_AUTO_RESET) && !io->episode) return B200ENV_ENULL;
    // Small batches (config #2: 65,536 instances = 512 blocks of 128 on 148 SMs, 3.46 blocks per SM -> the SMs that get
    // a 4th block set the time): halve the block until the grid has >= 8 blocks per SM so that the tail is <= 1 / 8
    int block = B200_BLOCK;
    const int64_t want = (int64_t)b200_persistent_grid((int64_t)1 << 40, 8, 32);
    while (block > 32 && (n + block - 1) / block < want) block >>= 1;
    B200_LAUNCH_TIO(cartpole_step_kernel, b200_grid(n, block), block, s, p, *io, n, flags, seed, off);
    return b200_check_launch();
}

int cartpole_rollout(int dtype, int64_t n, const void *params, const b200env_io *io, const b200env_rollout_spec *rs,
                     uint32_t flags, uint64_t seed, int64_t off, cudaStream_t s) {
    const b200_cartpole_params &p = *static_cast<const b200_cartpole_params *>(params);
    if (p.variant < 0 || p.variant > 2) return B200ENV_EENV;
    if (!io->state || !io->time || !io->action || !io->next_obs || !io->reward || !io->done || !io->flag)
        return B200ENV_ENULL;
    if ((flags & B200ENV_AUTO_RESET) && !io->episode) return B200ENV_ENULL;
    // one launch for the whole rollout: the grid is sized for latency hiding, not for a short tail -- 32-thread blocks
    // spread a small batch over every SM sub-partition
    int block = B200_BLOCK;
    const int64_t want = (int64_t)b200_persistent_grid((int64_t)1 << 40, 8, 32);
    while (block > 32 && (n + block - 1) / block < want) block >>= 1;
    B200_LAUNCH_TIO(cartpole_rollout_kernel, b200_grid(n, block), block, s, p, *io, *rs, n, flags, seed, off);
    return b200_check_launch();
}

int cartpole_reset(int dtype, int64_t n, const void *params, const b200env_io *io, const uint8_t *mask,
                   uint64_t seed, int64_t off, cudaStream_t s) {
    const b200_cartpole_params &p = *static_cast<const b200_cartpole_params *>(params);
    if (p.variant < 0 || p.variant > 2) return B200ENV_EENV;
    if (!io->state || !io->time || !io->episode) return B200ENV_ENULL;
    B200_LAUNCH_TIO(cartpole_reset_kernel, b200_grid(n), B200_BLOCK, s, p, *io, n, mask, seed, off, 0);
    return b200_check_launch();
}

int cartpole_observe(int dtype, int64_t n, const void *params, const b200env_io *io, cudaStream_t s) {
    const b200_cartpole_params &p = *static_cast<const b200_cartpole_params *>(params);
    if (p.variant < 0 || p.variant > 2) return B200ENV_EENV;
    if (!io->state || !io->time || !io->next_obs) return B200ENV_ENULL;
    B200_LAUNCH_TIO(cartpole_reset_kernel, b200_grid(n), B200_BLOCK, s, p, *io, n, nullptr, 0, 0, 1);
    return b200_check_launch();
}
