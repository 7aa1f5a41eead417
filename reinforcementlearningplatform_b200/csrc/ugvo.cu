// ugvo.cu -- K-UGVO: batched UGVForwardObstacleAvoidance step with the 37-ray fake laser (sm_100a).
//
// Replaces environment/UGVForwardObstacleAvoidance/UGVForwardObstacleAvoidance.py:261-557 (collision_check,
// get_fake_laser, get_state, is_Terminal, get_reward, ode, rk44, step_update, reset) and map.py:65-80,120-174 (map
// generation), plus the PPO2/DPPO2 demo copies (variant 1).  97 % of the reference's step time is the ray cast, run
// twice per step (before and after the RK4 update).
//
// Step kernel: block-cooperative, 64 instances per 128-thread block.  The scalar part of the step (unicycle RK4,
// collision test, centre-distance ordering of the obstacles, terminal flag, reward) runs one THREAD per instance; the
// rays of all instances of the block are then dealt to all threads, so every lane casts a ray (the first version ran
// one warp per instance: 37 of 64 lanes busy in the scan and all scalar work repeated by 32 lanes -- 3400 warp
// instructions per step, ncu profiles/r1/ugvo_kernel_ncu_v1_keys.txt).  Per pose only the obstacles within laser
// range are kept, in np.argsort(centre distance) order; a ray walks that list and stops at the FIRST obstacle it
// accepts -- the reference's selection rule (note N8: first accepted obstacle in centre-distance order, not the
// nearest crossing).  Reset / observe and the in-step auto-reset run one warp per instance: warp votes implement the
// lane-parallel rejection sampling of the obstacle map (64 candidates per round, two per lane; the lowest legal index
// wins, so the result is identical to trying the candidates one by one).
#define B200_SOA_INDEX // see common.cuh: the index form is faster for this warp-cooperative kernel
#include "common.cuh"

namespace {

typedef b200_ugvo_params P;
constexpr int MAXO = B200_UGVO_MAX_OBS;
constexpr int WARPS = 4; // per block: 4 consecutive instances share the 32-byte sectors of the SoA arrays
constexpr unsigned FULL = 0xffffffffu;

template <typename T> __device__ __forceinline__ T shfl(T v, int src);
template <> __device__ __forceinline__ double shfl<double>(double v, int src) { return __shfl_sync(FULL, v, src); }
template <> __device__ __forceinline__ float shfl<float>(float v, int src) { return __shfl_sync(FULL, v, src); }

template <typename T>
__device__ __forceinline__ T norm2(T a, T b) { return np_norm2<T>(a, b); }   // np.linalg.norm / dis_two_points, common.cuh

// utils/functions.py:35-46
template <typename T>
__device__ __forceinline__ T vector_rad(T x1, T y1, T x2, T y2) {
    const T n1 = norm2(x1, y1), n2 = norm2(x2, y2);
    if (n2 < (T)1e-4 || n1 < (T)1e-4) return (T)0;
    const T c = Mth<T>::min(Mth<T>::max((x1 * x2 + y1 * y2) / (n1 * n2), (T)-1), (T)1);
    return Mth<T>::acos(c);
}
// `cal_vector_rad(v1, v2) > pi / 2` without the acos: true iff the clamped cosine is negative (acos is decreasing and
// acos(c) rounds to a double above fl(pi/2) exactly when c < -5e-17; the band (-5e-17, 0) is unreachable in practice)
template <typename T>
__device__ __forceinline__ bool vector_rad_obtuse(T x1, T y1, T x2, T y2) {
    const T n1 = norm2(x1, y1), n2 = norm2(x2, y2);
    if (n2 < (T)1e-4 || n1 < (T)1e-4) return false;
    return (x1 * x2 + y1 * y2) / (n1 * n2) < (T)0;
}
// utils/functions.py:49-60
template <typename T>
__device__ __forceinline__ T vector_rad_oriented(T x1, T y1, T x2, T y2) {
    if (norm2(x2, y2) < (T)1e-4 || norm2(x1, y1) < (T)1e-4) return (T)0;
    return Mth<T>::atan2(x1 * y2 - y1 * x2, x1 * x2 + y1 * y2);
}

template <typename T>
struct Pose {
    T x, y, phi;
    T th1, th2, th3, th4; // bearings of the four map corners (:304-309)
    bool collided;        // collision_check() :261-272 -> every ray returns laserBlind
};

// In-range obstacle list of one pose.  `dis > laserDis + r0` (:349-351) is the same for every ray of a pose, so it is
// evaluated once per obstacle and the rays walk the compacted list (typically 3-5 of the 15 circles), kept in
// centre-distance order (np.argsort :301; ties: lower index first).  Element j lives at ptr[j * stride]: stride 1 for
// the warp-cooperative path (reset / observe), stride G for the block-cooperative step kernel ([slot][instance]).
template <typename T>
struct ObsList {
    const T *x0, *y0, *r0, *d;
    int stride, count;
};

// bearings of the four map corners seen from (x, y), :304-309
template <typename T>
__device__ __forceinline__ T corner_bearing(const P &p, T x, T y, int k) {
    const T vx = (k == 0 || k == 3) ? (T)p.map_x - x : (T)0 - x;
    const T vy = (k == 0 || k == 1) ? (T)p.map_y - y : (T)0 - y;
    const T th = vector_rad<T>((T)1, (T)0, vx, vy);
    return k < 2 ? th : -th;
}

// One ray of get_fake_laser (:302-395) for pose q; ray index in [0, n_rays).  No warp-level operations: lanes of one
// warp may belong to different instances.
template <typename T>
__device__ __forceinline__ T cast_ray(const P &p, const Pose<T> &q, int ray, const ObsList<T> &so) {
    const T LD = (T)p.laser_dis, LB = (T)p.laser_blind;
    if (q.collided) return LB; // collision_check() :261-272 -> every ray returns laserBlind
    const T x = q.x, y = q.y, xm = (T)p.map_x, ym = (T)p.map_y;
    // np.linspace(phi - R, phi + R, n): arange * step + start, last element = stop
    const T a0 = q.phi - (T)p.laser_range, a1 = q.phi + (T)p.laser_range;
    const T nm1 = (T)(p.n_rays - 1);
    const T step = Divisor<T>(nm1, Mth<T>::rcp(nm1)).div(a1 - a0);
    T phi = (ray == p.n_rays - 1) ? a1 : (T)ray * step + a0;
    if (phi > (T)M_PI) phi -= (T)(2 * M_PI);
    if (phi < (T)-M_PI) phi += (T)(2 * M_PI);
    T sphi, cphi;
    Mth<T>::sincos(phi, &sphi, &cphi);
    const T m = Mth<T>::div(sphi, cphi); // np.tan(phi) :311 (constant-bank sincos + rcp-based quotient, <= 2.5 ulp)
    const T b = y - m * x;
    const T m2p1 = m * m + (T)1;
    const T sq = Mth<T>::sqrt(m2p1);
    const Divisor<T> dsq(sq, Mth<T>::rcp(sq)), dm2(m2p1, Mth<T>::rcp(m2p1));
    const T am = Mth<T>::abs(m);
    const T cosT = dsq.div(am), sinT = dsq.r; // |m| / sqrt(m^2 + 1), 1 / sqrt(m^2 + 1)
    const T ld_sq = dsq.div(LD);               // laserDis / sqrt(m^2 + 1)
    const bool mpos = m >= (T)0;
    T tx, ty; // end point of the ray on the map border or at laserDis (:313-343)
    if (q.th4 < phi && phi <= q.th1) { // right wall
        tx = xm; ty = m * xm + b;
        const T t = x + ld_sq;
        if (t < xm) { tx = t; ty = mpos ? y + cosT * LD : y - cosT * LD; }
    } else if (q.th1 < phi && phi <= q.th2) { // top wall
        if (am < (T)1e8) { tx = (ym - b) / m; ty = ym; } else { tx = x; ty = ym; }
        const T t = y + dsq.div(am * LD);
        if (t < ym) { ty = t; tx = mpos ? x + LD * sinT : x - LD * sinT; }
    } else if (q.th3 < phi && phi <= q.th4) { // bottom wall
        if (am < (T)1e8) { tx = -b / m; ty = (T)0; } else { tx = x; ty = (T)0; }
        const T t = y - dsq.div(am * LD);
        if (t > (T)0) { ty = t; tx = mpos ? x - LD * sinT : x + LD * sinT; }
    } else { // left wall
        tx = (T)0; ty = b;
        const T t = x - ld_sq;
        if (t > (T)0) { tx = t; ty = mpos ? y - cosT * LD : y + cosT * LD; }
    }
    const T rdx = tx - x, rdy = ty - y;
    const T sg = rdx > (T)0 ? (T)1 : (rdx < (T)0 ? (T)-1 : (T)0);
    const T lo = Mth<T>::min(x, tx), hi = Mth<T>::max(x, tx);
    const T ray_len = norm2(rdx, rdy);
    const bool ray_ok = !(ray_len < (T)1e-4); // cal_vector_rad returns 0 for a degenerate ray (never > pi/2)
    for (int j = 0; j < so.count; ++j) { // in-range obstacles in centre-distance order, first accepted wins (N8)
        const int o = j * so.stride;
        const T x0 = so.x0[o], y0 = so.y0[o], r0 = so.r0[o];
        const T dj = so.d[o]; // = |centre - start|, the second norm of cal_vector_rad
        // `abs(m x0 - y0 + b) / sqrt(m^2 + 1) > r0` (:353): decided on the product form; the exact quotient is only
        // evaluated when the two sides are within a few ulp of each other (same decision as the reference, no division)
        const T num = Mth<T>::abs(m * x0 - y0 + b), rhs = r0 * sq;
        bool miss = num > rhs;
        if (Mth<T>::abs(num - rhs) <= (T)(sizeof(T) == 8 ? 1e-15 : 1e-6) * rhs) miss = num / sq > r0;
        // cal_vector_rad(ray, centre - start) > pi / 2  <=>  both vectors non-degenerate and their dot product < 0
        // (dividing by the positive norms and taking acos cannot change the sign; see vector_rad_obtuse)
        if (miss) continue; // most in-range circles are missed: the obtuse-angle test is only made for the others
        const bool behind = ray_ok && !(dj < (T)1e-4) && (rdx * (x0 - x) + rdy * (y0 - y) < (T)0);
        if (!behind) {
            const T fx = dm2.div(x0 + m * y0 - m * b);
            const T fy = dm2.div(m * x0 + m * m * y0 + b);
            const T rd = norm2(fx - x0, fy - y0);
            const T cross = fx - dsq.div(sg * Mth<T>::sqrt(r0 * r0 - rd * rd)); // NaN (no crossing) fails the test below
            if (lo <= cross && cross <= hi) {
                const T dis = Mth<T>::abs(cross - x) * sq;
                return dis < LB ? LB : dis;
            }
        }
    }
    // no obstacle hit (:382-395): ray_len = norm2(x - tx, y - ty) (the squares are sign-symmetric)
    if (ray_len > LD) return LD;
    if (LB < ray_len && ray_len <= LD) return ray_len;
    return LB;
}

// ---- warp-cooperative pose preparation (reset / observe path): lane k < nobs owns obstacle k (cx, cy, r)
// (sx0, sy0, sr0, sd: MAXO elements each in shared memory, owned by this warp)
template <typename T>
__device__ __forceinline__ ObsList<T> prepare_pose_warp(const P &p, Pose<T> &q, int lane, int nobs, T cx, T cy, T r,
                                                        T *sx0, T *sy0, T *sr0, T *sd) {
    const bool mine = lane < nobs;
    const T d = mine ? norm2(q.x - cx, q.y - cy) : (T)1e300;
    q.collided = __any_sync(FULL, mine && d <= r + (T)p.r_vehicle);
    const bool inr = mine && !(d > (T)p.laser_dis + r); // :349 `if dis > self.laserDis + _r: continue`
    const unsigned in_mask = __ballot_sync(FULL, inr);
    int rank = 0; // number of in-range obstacles strictly closer (ties: lower index first) -- np.argsort order
    for (unsigned mm = in_mask; mm; mm &= mm - 1) {
        const int j = __ffs(mm) - 1;
        const T dj = shfl<T>(d, j);
        rank += (dj < d || (dj == d && j < lane));
    }
    if (inr) { sx0[rank] = cx; sy0[rank] = cy; sr0[rank] = r; sd[rank] = d; }
    T th = (T)0;
    if (lane < 4) th = corner_bearing<T>(p, q.x, q.y, lane);
    q.th1 = shfl<T>(th, 0); q.th2 = shfl<T>(th, 1); q.th3 = shfl<T>(th, 2); q.th4 = shfl<T>(th, 3);
    __syncwarp();
    ObsList<T> l;
    l.x0 = sx0; l.y0 = sy0; l.r0 = sr0; l.d = sd; l.stride = 1; l.count = __popc(in_mask);
    return l;
}

struct Draw2 { double u0, u1; };
__device__ __forceinline__ Draw2 draw2(uint64_t seed, uint64_t gid, uint32_t ep, uint32_t block) {
    Philox g(seed, gid, ep);
    g.c3 = block;
    g.block();
    Draw2 d;
    d.u0 = ((double)(g.r[0] >> 5) * 67108864.0 + (double)(g.r[1] >> 6)) * (1.0 / 9007199254740992.0);
    d.u1 = ((double)(g.r[2] >> 5) * 67108864.0 + (double)(g.r[3] >> 6)) * (1.0 / 9007199254740992.0);
    return d;
}
// One block per obstacle candidate: the centre takes the 2 x 53 high bits like draw2, the radius the 22 bits draw2 throws
// away (5 + 6 + 5 + 6 low bits of the four words) -- a U[0, 1) with 2^-22 resolution for a radius drawn from
// [r_min, r_max].  A candidate used to cost two Philox blocks (220 of its ~330 instructions); the oracle draws the same.
struct Draw3 { double u0, u1, u2; };
__device__ __forceinline__ Draw3 draw3(uint64_t seed, uint64_t gid, uint32_t ep, uint32_t block) {
    Philox g(seed, gid, ep);
    g.c3 = block;
    g.block();
    Draw3 d;
    d.u0 = ((double)(g.r[0] >> 5) * 67108864.0 + (double)(g.r[1] >> 6)) * (1.0 / 9007199254740992.0);
    d.u1 = ((double)(g.r[2] >> 5) * 67108864.0 + (double)(g.r[3] >> 6)) * (1.0 / 9007199254740992.0);
    const uint32_t low = ((g.r[0] & 31u) << 17) | ((g.r[1] & 63u) << 11) | ((g.r[2] & 31u) << 6) | (g.r[3] & 63u);
    d.u2 = (double)low * (1.0 / 4194304.0);
    return d;
}
__device__ __forceinline__ double lerp_u(double lo, double hi, double u) { return ::fma(hi - lo, u, lo); }
// dis_two_points(a, b) <= R, i.e. sqrt(dx^2 + dy^2) <= R (map.py:122,131-133), decided on the squares; the square root is
// only taken when the two sides agree to ~14 digits, so the decision is the reference's in every case
__device__ __forceinline__ bool within(double dx, double dy, double R) {
    const double d2 = ::fma(dy, dy, dx * dx), R2 = R * R;   // the squared np.linalg.norm (common.cuh np_norm2)
    if (fabs(d2 - R2) <= 1e-13 * R2) return sqrt(d2) <= R;
    return d2 <= R2;
}

// reset(random=True) :527-557 + Map.generate_circle_obs_training (map.py:152-174), cooperative over the warp.
// Outputs (uniform over the warp): start/target/phi0; per-lane obstacle k = lane (cx, cy, r), nobs.
// `pl`: 3 * MAXO doubles of shared memory owned by this warp (x, y, r of the obstacles placed so far): the legality loop
// reads them as broadcasts, UGVO_PLACED_GROUP obstacles per vote (measured: a wash against one shuffle-broadcast and one
// vote per obstacle -- larger groups lose more to the delayed early exit than they win in latency).
__device__ __forceinline__ void reset_map(const P &p, uint64_t seed, uint64_t gid, uint32_t ep, int lane, double *pl, double &sx,
                                          double &sy, double &tx, double &ty, double &phi0, double &ocx, double &ocy,
                                          double &orr, int &nobs) {
    const double lo = p.st_margin, hx = p.map_x - p.st_margin, hy = p.map_y - p.st_margin;
    Draw2 d = draw2(seed, gid, ep, 0);
    sx = lerp_u(lo, hx, d.u0);
    sy = lerp_u(lo, hy, d.u1);
    // target: first candidate (blocks 1..64) at least safety_dis_st away; 32 candidates per round
    tx = sx; ty = sy;
    for (int round = 0; round < 2; ++round) {
        d = draw2(seed, gid, ep, 1u + (uint32_t)(round * 32 + lane));
        const double cx = lerp_u(lo, hx, d.u0), cy = lerp_u(lo, hy, d.u1);
        const bool ok = !(sqrt(::fma(cy - sy, cy - sy, (cx - sx) * (cx - sx))) < p.safety_dis_st);
        const unsigned m = __ballot_sync(FULL, ok);
        if (m) {
            const int src = __ffs(m) - 1;
            tx = __shfl_sync(FULL, cx, src);
            ty = __shfl_sync(FULL, cy, src);
            break;
        }
        if (round == 1) { // no candidate accepted: the oracle keeps the last one drawn (block 64)
            tx = __shfl_sync(FULL, cx, 31);
            ty = __shfl_sync(FULL, cy, 31);
        }
    }
    ocx = 0.0; ocy = 0.0; orr = 0.0;
    nobs = 0;
    const int want = p.obs_num < MAXO ? p.obs_num : MAXO;
    // Rounds of 32 * NC candidates, NC per lane (indices 32 NC r + 32 j + lane): the NC Philox blocks and legality chains
    // of a lane are independent, which shortens the dependent-instruction path of a placement (the reset launch is
    // latency-bound: ~8 warps per SM alive on average; NC = 2: 0.874 -> 0.819 ms per step at the steady-state reset rate).
    // The winner is still the lowest legal candidate index, so the map does not depend on NC.
#ifndef UGVO_CAND_PER_LANE
#define UGVO_CAND_PER_LANE 2
#endif
#ifndef UGVO_PLACED_GROUP
#define UGVO_PLACED_GROUP 2 // 1-vote-per-obstacle shuffles 0.766, groups of 2 / 4 / 8 / 15 from shared memory 0.758 / 0.775 / 0.792 / 0.804 ms per step
#endif
    constexpr int NC = UGVO_CAND_PER_LANE;
    for (int k = 0; k < want; ++k) {
        bool placed = false;
        for (int round = 0; round < 64 / NC && !placed; ++round) {
            const uint32_t blk = 1000u + 2048u * (uint32_t)k + (uint32_t)(round * 32 * NC + lane);
            double cx[NC], cy[NC], r[NC];
            bool legal[NC]; // map.py:129-139
#pragma unroll
            for (int j = 0; j < NC; ++j) {
                const Draw3 dc = draw3(seed, gid, ep, blk + 32u * (uint32_t)j);
                cx[j] = lerp_u(0., p.map_x, dc.u0); cy[j] = lerp_u(0., p.map_y, dc.u1); r[j] = lerp_u(p.r_min, p.r_max, dc.u2);
            }
#pragma unroll
            for (int j = 0; j < NC; ++j)
                legal[j] = !within(sx - cx[j], sy - cy[j], r[j] + p.safety_dis_st) &&
                           !within(tx - cx[j], ty - cy[j], r[j] + p.safety_dis_st);
            for (int q0 = 0; q0 < nobs; q0 += UGVO_PLACED_GROUP) { // placed obstacles, a group per vote
                bool any = false;
#pragma unroll
                for (int j = 0; j < NC; ++j) any = any || legal[j];
                if (!__any_sync(FULL, any)) break; // all candidates of this round are already rejected
#pragma unroll
                for (int g = 0; g < UGVO_PLACED_GROUP; ++g) {
                    const int q = q0 + g;
                    if (q < nobs) {
                        const double qx = pl[q], qy = pl[MAXO + q], qr = pl[2 * MAXO + q];
#pragma unroll
                        for (int j = 0; j < NC; ++j)
                            if (within(qx - cx[j], qy - cy[j], qr + r[j] + p.safety_dis_obs)) legal[j] = false;
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < NC; ++j) {
                const unsigned m = __ballot_sync(FULL, legal[j]);
                if (m && !placed) {
                    const int src = __ffs(m) - 1;
                    const double wx = __shfl_sync(FULL, cx[j], src), wy = __shfl_sync(FULL, cy[j], src);
                    const double wr = __shfl_sync(FULL, r[j], src);
                    if (lane == nobs) { ocx = wx; ocy = wy; orr = wr; pl[nobs] = wx; pl[MAXO + nobs] = wy; pl[2 * MAXO + nobs] = wr; }
                    ++nobs;
                    placed = true;
                    __syncwarp();
                }
            }
        }
        if (!placed) break;
    }
    d = draw2(seed, gid, ep, 100);
    phi0 = lerp_u(-M_PI, M_PI, d.u0);
}

enum { F_X = 0, F_Y, F_VEL, F_PHI, F_OMEGA, F_TX, F_TY, F_NOBS, F_OBS };

// get_state :399-411, kinematic part (4 terms) of pose (x, y, phi) with velocity / rate (vel, omega)
template <typename T>
__device__ __forceinline__ void kin_obs(const P &p, T x, T y, T vel, T phi, T omega, T tgx, T tgy, T *o, T *err_out,
                                        T *ephi_out) {
    T s, c;
    Mth<T>::sincos(phi, &s, &c);
    const T g = (T)p.static_gain;
    const T e = norm2(tgx - x, tgy - y), ephi = vector_rad_oriented<T>(c, s, tgx - x, tgy - y);
    o[0] = ((T)(2 / p.e_max) * e - (T)1) * g;
    o[1] = ((T)(2 / p.v_max) * vel - (T)1) * g;
    o[2] = ephi / (T)p.e_phi_max * g;
    o[3] = omega / (T)p.omega_max * g;
    if (err_out) *err_out = e;
    if (ephi_out) *ephi_out = ephi;
}

// ---- warp view of one instance (reset / observe path): scalars are warp-uniform, lane k holds obstacle k
template <typename T>
struct WarpInst {
    T x, y, vel, phi, omega, tgx, tgy, ocx, ocy, orr;
    int nobs;
    double time;
};

template <typename T>
__device__ __forceinline__ void warp_load(const b200env_io &io, int64_t n, int64_t i, int lane, WarpInst<T> &e) {
    T sc = (T)0; // lanes 0..7 fetch the scalar fields, lane k the k-th obstacle; scalars are broadcast
    if (lane < F_OBS) sc = ld<T>(io.state, n, lane, i);
    e.x = shfl<T>(sc, F_X); e.y = shfl<T>(sc, F_Y); e.vel = shfl<T>(sc, F_VEL); e.phi = shfl<T>(sc, F_PHI);
    e.omega = shfl<T>(sc, F_OMEGA); e.tgx = shfl<T>(sc, F_TX); e.tgy = shfl<T>(sc, F_TY);
    e.nobs = (int)shfl<T>(sc, F_NOBS);
    e.ocx = e.ocy = e.orr = (T)0;
    if (lane < MAXO) {
        e.ocx = ld<T>(io.state, n, F_OBS + 3 * lane + 0, i);
        e.ocy = ld<T>(io.state, n, F_OBS + 3 * lane + 1, i);
        e.orr = ld<T>(io.state, n, F_OBS + 3 * lane + 2, i);
    }
    e.time = io.time[i];
}

// reset(random=True) :527-557 of instance i by one warp; writes the whole persistent state
template <typename T>
__device__ __forceinline__ void warp_reset(const P &p, const b200env_io &io, int64_t n, int64_t i, uint64_t seed,
                                           int64_t off, int lane, double *pl, WarpInst<T> &e) {
    const uint32_t ep = io.episode[i];
    double sx, sy, ttx, tty, phi0, cx, cy, rr;
    int no;
    reset_map(p, seed, (uint64_t)(off + i), ep, lane, pl, sx, sy, ttx, tty, phi0, cx, cy, rr, no);
    e.x = (T)sx; e.y = (T)sy; e.tgx = (T)ttx; e.tgy = (T)tty; e.phi = (T)phi0; e.vel = (T)0; e.omega = (T)0;
    e.ocx = (T)cx; e.ocy = (T)cy; e.orr = (T)rr; e.nobs = no;
    e.time = 0.0;
    __syncwarp();
    if (lane == 0) {
        io.episode[i] = ep + 1u;
        st<T>(io.state, n, F_X, i, e.x); st<T>(io.state, n, F_Y, i, e.y); st<T>(io.state, n, F_VEL, i, e.vel);
        st<T>(io.state, n, F_PHI, i, e.phi); st<T>(io.state, n, F_OMEGA, i, e.omega);
        st<T>(io.state, n, F_TX, i, e.tgx); st<T>(io.state, n, F_TY, i, e.tgy); st<T>(io.state, n, F_NOBS, i, (T)e.nobs);
        io.time[i] = 0.0;
    }
    if (lane < MAXO) {
        st<T>(io.state, n, F_OBS + 3 * lane + 0, i, e.ocx);
        st<T>(io.state, n, F_OBS + 3 * lane + 1, i, e.ocy);
        st<T>(io.state, n, F_OBS + 3 * lane + 2, i, e.orr);
    }
}

// get_state :399-411 of instance i by one warp (lanes = rays) into dst[41][n]
template <typename T, bool IO32>
__device__ __forceinline__ void warp_observe(const P &p, int64_t n, int64_t i, int lane, const WarpInst<T> &e, void *dst,
                                             T *sx0, T *sy0, T *sr0, T *sd) {
    Pose<T> q;
    q.x = e.x; q.y = e.y; q.phi = e.phi;
    __syncwarp();
    const ObsList<T> l = prepare_pose_warp<T>(p, q, lane, e.nobs, e.ocx, e.ocy, e.orr, sx0, sy0, sr0, sd);
    const T g = (T)p.static_gain;
    for (int ray = lane; ray < p.n_rays; ray += 32)
        stio<T, IO32>(dst, n, 4 + ray, i, ((T)2 * cast_ray<T>(p, q, ray, l) / (T)p.laser_dis - (T)1) * g);
    if (lane == 0) {
        T o[4];
        kin_obs<T>(p, e.x, e.y, e.vel, e.phi, e.omega, e.tgx, e.tgy, o, nullptr, nullptr);
#pragma unroll
        for (int k = 0; k < 4; ++k) stio<T, IO32>(dst, n, k, i, o[k]);
    }
    __syncwarp();
}

// reset (mode 1, masked) / observe (mode 2): one warp per instance
template <typename T, bool IO32>
__global__ void __launch_bounds__(WARPS * 32)
ugvo_aux_kernel(const __grid_constant__ P p, const __grid_constant__ b200env_io io, int64_t n, uint64_t seed,
                int64_t off, const uint8_t *mask, int mode) {
    __shared__ T s_o[WARPS][4][MAXO];
    __shared__ double s_pl[WARPS][3 * MAXO];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t i = (int64_t)blockIdx.x * WARPS + w;
    if (i >= n) return; // whole warp exits together
    if (mode == 1 && mask && !mask[i]) return;
    WarpInst<T> e;
    warp_load<T>(io, n, i, lane, e);
    if (mode == 1) warp_reset<T>(p, io, n, i, seed, off, lane, s_pl[w], e);
    if (io.next_obs) warp_observe<T, IO32>(p, n, i, lane, e, io.next_obs, s_o[w][0], s_o[w][1], s_o[w][2], s_o[w][3]);
}

// ---- step: block-cooperative.  G instances per block.
//   phase 1  thread t = instance t: unicycle RK4 (rk44 :482-501), collision test, in-range obstacle list of the pose
//            (insertion sort by centre distance into shared memory, [slot][instance] so thread t stays in bank t),
//            corner bearings, terminal flag, reward, kinematic observation terms -- all scalar work of the step is done
//            once per instance with every lane busy, and its loads / stores are coalesced over instances;
//   phase 2  the G x n_rays rays are dealt round-robin to all threads of the block (a warp covers at most two
//            instances, so the obstacle lists are shared-memory broadcasts) -- every lane casts a ray;
//   (phase 3, auto-reset of the terminated instances, is a second launch: ugvo_autoreset_kernel)
// With io.obs == NULL (observation reuse, vec_env.py) only the post-update scan is cast (SURVEY 8d: one scan per step).
#ifndef UGVO_G
#define UGVO_G 64
#endif
#ifndef UGVO_TPB
#define UGVO_TPB 128
#endif
// six resident blocks per SM (80 registers, the 36.7 KB of shared memory per block allow no more): the ray loop is a
// chain of dependent fp64 operations, and 24 warps hide it better than the 16 of the uncapped 120-register build
// (0.942 -> 0.863 ms per step of 262,144 instances at the steady-state reset rate, A/B on one box)
#ifndef UGVO_MINB
#define UGVO_MINB 6
#endif
constexpr int G = UGVO_G;
constexpr int TPB = UGVO_TPB;
static_assert(TPB >= G, "phase 1 runs one thread per instance");

template <typename T, bool IO32>
__global__ void __launch_bounds__(TPB, UGVO_MINB)
ugvo_step_kernel(const __grid_constant__ P p, const __grid_constant__ b200env_io io, int64_t n, uint32_t flags,
                 uint64_t seed, int64_t off) {
    __shared__ T s_o[4][MAXO][G];                 // x0, y0, r0, d of the in-range obstacles, [slot][instance]
    __shared__ T s_pose[7][G];                    // x, y, phi, th1..th4
    __shared__ int s_cnt[G];
    __shared__ unsigned char s_col[G], s_mirror[G];
    const int t = threadIdx.x;
    const int64_t base = (int64_t)blockIdx.x * G;
    const int gv = (int)((n - base) < (int64_t)G ? (n - base) : (int64_t)G);
    const int NR = p.n_rays;
    const bool own = t < gv;
    const int64_t i = base + t;
    const bool scan_a = io.obs != nullptr;
    const T g = (T)p.static_gain;
    T x = (T)0, y = (T)0, vel = (T)0, phi = (T)0, omega = (T)0, tgx = (T)0, tgy = (T)0;
    T xa = (T)0, ya = (T)0, phia = (T)0, cur_e = (T)0, cur_vel = (T)0;
    int nobs = 0;
    double time = 0.0;
    if (own) {
        x = ld<T>(io.state, n, F_X, i); y = ld<T>(io.state, n, F_Y, i); vel = ld<T>(io.state, n, F_VEL, i);
        phi = ld<T>(io.state, n, F_PHI, i); omega = ld<T>(io.state, n, F_OMEGA, i);
        tgx = ld<T>(io.state, n, F_TX, i); tgy = ld<T>(io.state, n, F_TY, i);
        nobs = (int)ld<T>(io.state, n, F_NOBS, i);
        time = io.time[i];
        const T a_lin = ldio<T, IO32>(io.action, n, 0, i), a_ang = ldio<T, IO32>(io.action, n, 1, i);
        xa = x; ya = y; phia = phi; cur_vel = vel;
        // ---- step_update :510-520: current_state = get_state() (kinematic part; the laser part is scan A)
        if (scan_a) {
            T o[4];
            kin_obs<T>(p, x, y, vel, phi, omega, tgx, tgy, o, nullptr, nullptr);
#pragma unroll
            for (int k = 0; k < 4; ++k) stio<T, IO32>(io.obs, n, k, i, o[k]);
            cur_e = o[0];
        } else {
            cur_e = ((T)(2 / p.e_max) * norm2(tgx - x, tgy - y) - (T)1) * g; // current_state[0] (demo-copy reward)
        }
        // ---- rk44 :482-501 / demo copy :488-509
        const T h = (T)p.dt, half = (T)0.5, kf = (T)p.kf, kt = (T)p.kt;
        T s, c;
        Mth<T>::sincos(phi, &s, &c);
        const T k1x = h * (vel * c), k1y = h * (vel * s), k1v = h * (a_lin - kf * vel), k1p = h * omega, k1o = h * (a_ang - kt * omega);
        const T v2 = vel + k1v * half, o2 = omega + k1o * half;
        Mth<T>::sincos(phi + k1p * half, &s, &c);
        const T k2x = h * (v2 * c), k2y = h * (v2 * s), k2v = h * (a_lin - kf * v2), k2p = h * o2, k2o = h * (a_ang - kt * o2);
        const T v3 = vel + k2v * half, o3 = omega + k2o * half;
        Mth<T>::sincos(phi + k2p * half, &s, &c);
        const T k3x = h * (v3 * c), k3y = h * (v3 * s), k3v = h * (a_lin - kf * v3), k3p = h * o3, k3o = h * (a_ang - kt * o3);
        const T v4 = vel + k3v, o4 = omega + k3o;
        Mth<T>::sincos(phi + k3p, &s, &c);
        const T k4x = h * (v4 * c), k4y = h * (v4 * s), k4v = h * (a_lin - kf * v4), k4p = h * o4, k4o = h * (a_ang - kt * o4);
        const T nx = x + div6<T>(k1x + (T)2 * k2x + (T)2 * k3x + k4x);
        const T ny = y + div6<T>(k1y + (T)2 * k2y + (T)2 * k3y + k4y);
        const T nv = vel + div6<T>(k1v + (T)2 * k2v + (T)2 * k3v + k4v);
        const T np_ = phi + div6<T>(k1p + (T)2 * k2p + (T)2 * k3p + k4p);
        const T no = omega + div6<T>(k1o + (T)2 * k2o + (T)2 * k3o + k4o);
        if (p.variant == 0) {
            x = nx; y = ny; vel = nv; phi = np_; omega = no;
            if (vel < (T)0) vel = (T)0;
        } else if (vel < (T)0) { // the PRE-update velocity is tested (note N9): pose frozen
            phi = np_; omega = no; vel = (T)0;
        } else {
            x = nx; y = ny; vel = nv; phi = np_; omega = no;
        }
        time += p.dt;
        if (phi > (T)M_PI) phi -= (T)(2 * M_PI);
        if (phi < (T)-M_PI) phi += (T)(2 * M_PI);
    }

    for (int scan = scan_a ? 0 : 1; scan < 2; ++scan) {
        if (own) {
            const T px = scan ? x : xa, py = scan ? y : ya, pphi = scan ? phi : phia;
            // collision_check :261-272 + in-range list in np.argsort(centre distance) order (stable insertion)
            bool collided = false;
            int cnt = 0;
            for (int k = 0; k < nobs; ++k) {
                const T cx = ld<T>(io.state, n, F_OBS + 3 * k + 0, i), cy = ld<T>(io.state, n, F_OBS + 3 * k + 1, i);
                const T r = ld<T>(io.state, n, F_OBS + 3 * k + 2, i);
                const T d = norm2(px - cx, py - cy);
                collided = collided || d <= r + (T)p.r_vehicle;
                if (!(d > (T)p.laser_dis + r)) { // :349 `if dis > self.laserDis + _r: continue`
                    int pos = cnt;
                    while (pos > 0 && s_o[3][pos - 1][t] > d) {
#pragma unroll
                        for (int a = 0; a < 4; ++a) s_o[a][pos][t] = s_o[a][pos - 1][t];
                        --pos;
                    }
                    s_o[0][pos][t] = cx; s_o[1][pos][t] = cy; s_o[2][pos][t] = r; s_o[3][pos][t] = d;
                    ++cnt;
                }
            }
            s_cnt[t] = cnt;
            s_col[t] = collided ? 1 : 0;
            s_pose[0][t] = px; s_pose[1][t] = py; s_pose[2][t] = pphi;
#pragma unroll
            for (int k = 0; k < 4; ++k) s_pose[3 + k][t] = corner_bearing<T>(p, px, py, k);
            if (scan == 1) {
                // ---- is_Terminal :431-449
                T nk[4], err, ephi;
                kin_obs<T>(p, x, y, vel, phi, omega, tgx, tgy, nk, &err, &ephi);
                const bool succ = Mth<T>::abs(err) <= (T)0.05 && (p.variant != 0 || Mth<T>::abs(omega) < (T)0.01) &&
                                  Mth<T>::abs(vel) < (T)0.01;
                int flag = 0;
                if (x > (T)p.map_x || x < (T)0 || y > (T)p.map_y || y < (T)0) flag = 1;
                if (time > p.time_max) flag = 2;
                if (succ) flag = 3;
                if (collided) flag = 4;
                const bool done = flag != 0;
                const bool will_reset = done && (flags & B200ENV_AUTO_RESET);
                // ---- get_reward :451-467 / demo copy :449-473
                T reward;
                if (p.variant == 0) {
                    const T u_pos = -Mth<T>::abs(err) * (T)p.Q_pos, u_vel = -Mth<T>::abs(vel) * (T)p.Q_vel;
                    const T u_phi = err > (T)0.1 ? -Mth<T>::abs(ephi) * (T)p.Q_phi : (T)0;
                    const T u_omega = -Mth<T>::abs(omega) * (T)p.Q_omega;
                    T u_psi = (T)0;
                    if (flag == 1) u_psi = (T)((p.time_max - time) / p.dt) * (u_pos + u_vel + u_phi + u_omega);
                    reward = u_pos + u_vel + u_phi + u_omega + u_psi;
                } else {
                    const T cur1 = ((T)(2 / p.v_max) * cur_vel - (T)1) * g;
                    const T r1 = (T)-1 - Mth<T>::abs(omega) * (T)0.1;
                    const T r2 = cur_e > nk[0] + (T)1e-3 ? (T)5 : ((T)1e-3 + cur_e < nk[0] ? (T)-5 : (T)0);
                    const T r3 = Mth<T>::abs(cur1) > Mth<T>::abs(nk[1]) + (T)1e-2 ? (T)2
                                 : ((T)1e-2 + Mth<T>::abs(cur1) < Mth<T>::abs(nk[1]) ? (T)-2 : (T)0);
                    const T r4 = succ ? (T)500 : (flag == 4 ? (T)-300 : (T)0);
                    reward = r1 + r2 + r3 + r4;
                }
                const bool mirror = !will_reset && io.reset_obs; // policy-facing obs = next_obs unless reset
                s_mirror[t] = mirror ? 1 : 0;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    stio<T, IO32>(io.next_obs, n, k, i, nk[k]);
                    if (mirror) stio<T, IO32>(io.reset_obs, n, k, i, nk[k]);
                }
                stio<T, IO32>(io.reward, n, 0, i, reward);
                io.done[i] = done ? 1 : 0;
                io.flag[i] = flag;
                if (will_reset) { // re-initialised by ugvo_autoreset_kernel
                    if (io.work) io.work[1 + atomicAdd(io.work, 1)] = (int32_t)i;
                } else {
                    st<T>(io.state, n, F_X, i, x); st<T>(io.state, n, F_Y, i, y); st<T>(io.state, n, F_VEL, i, vel);
                    st<T>(io.state, n, F_PHI, i, phi); st<T>(io.state, n, F_OMEGA, i, omega);
                    io.time[i] = time;
                }
            }
        }
        __syncthreads();
        // ---- phase 2: get_fake_laser :274-397 for all rays of the block
        void *dst = scan ? io.next_obs : io.obs;
        const int total = gv * NR;
        const Divisor<T> by_ld((T)p.laser_dis);
        for (int idx = t; idx < total; idx += TPB) {
            const int li = idx / NR, ray = idx - li * NR;
            Pose<T> q;
            q.x = s_pose[0][li]; q.y = s_pose[1][li]; q.phi = s_pose[2][li];
            q.th1 = s_pose[3][li]; q.th2 = s_pose[4][li]; q.th3 = s_pose[5][li]; q.th4 = s_pose[6][li];
            q.collided = s_col[li] != 0;
            ObsList<T> l;
            l.x0 = &s_o[0][0][li]; l.y0 = &s_o[1][0][li]; l.r0 = &s_o[2][0][li]; l.d = &s_o[3][0][li];
            l.stride = G; l.count = s_cnt[li];
            const T v = (by_ld.div((T)2 * cast_ray<T>(p, q, ray, l)) - (T)1) * g;
            stio<T, IO32>(dst, n, 4 + ray, base + li, v);
            if (scan && s_mirror[li]) stio<T, IO32>(io.reset_obs, n, 4 + ray, base + li, v);
        }
        __syncthreads();
    }
}

// ---- phase 3 of a step with B200ENV_AUTO_RESET (the `env.reset(True)` branch of the train loops) as its own launch:
// every warp looks at the `done` flags of 32 consecutive instances and re-initialises the terminated ones, one after
// the other, with all 32 lanes (map rejection sampling by ballot, then the 37-ray reset observation).  Kept out of the
// step kernel because a reset is ~3000 dependent warp instructions: inside the step it left three of the four warps of
// a block idle behind it (0.60 -> 0.95 ms per step at ~1 reset per block, ncu/bench).  With the optional scratch list
// io.work the step kernel appends the terminated instances and the warps of this grid take them one at a time from a
// ticket counter; without it every warp scans the `done` flags of its 32-instance groups.
constexpr int RESET_WARPS = 8;
#ifndef UGVO_RESET_MINB
#define UGVO_RESET_MINB 3 // 80 registers, no spills; 3 / 4 / 5 / 6 blocks per SM measured within 1 % of each other
#endif
template <typename T, bool IO32>
__global__ void __launch_bounds__(RESET_WARPS * 32, UGVO_RESET_MINB)
ugvo_autoreset_kernel(const __grid_constant__ P p, const __grid_constant__ b200env_io io, int64_t n, uint64_t seed,
                      int64_t off) {
    __shared__ T s_o[RESET_WARPS][4][MAXO];
    __shared__ double s_pl[RESET_WARPS][3 * MAXO];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int64_t gw = (int64_t)blockIdx.x * RESET_WARPS + w, nw = (int64_t)gridDim.x * RESET_WARPS;
    if (io.work) {
        // the step kernel appended the terminated instances to io.work[1..count].  A reset takes between ~15 and ~250
        // sampling rounds (crowded maps: half of them give up on one obstacle after 64 rounds), so dealing the list out in
        // equal shares left most warps idle behind the unlucky ones (warps active 12 % of peak under ncu); every warp now
        // takes the next entry when it is free -- work[0] is the ticket counter, counted down (it ends below zero; the
        // launcher clears it before every step kernel).
        for (;;) {
            int tk = 0;
            if (lane == 0) tk = atomicSub(io.work, 1);
            tk = __shfl_sync(FULL, tk, 0);
            if (tk <= 0) break;
            const int64_t ir = io.work[tk];
            WarpInst<T> e;
            warp_reset<T>(p, io, n, ir, seed, off, lane, s_pl[w], e);
            if (io.reset_obs) warp_observe<T, IO32>(p, n, ir, lane, e, io.reset_obs, s_o[w][0], s_o[w][1], s_o[w][2], s_o[w][3]);
        }
        return;
    }
    // no scratch list: every warp scans the `done` flags of 32-instance groups
    for (int64_t first = gw * 32; first < n; first += nw * 32) {
        const int64_t mine = first + lane;
        unsigned todo = __ballot_sync(FULL, mine < n && io.done[mine] != 0);
        while (todo) {
            const int64_t ir = first + (__ffs(todo) - 1);
            todo &= todo - 1;
            WarpInst<T> e;
            warp_reset<T>(p, io, n, ir, seed, off, lane, s_pl[w], e);
            if (io.reset_obs) warp_observe<T, IO32>(p, n, ir, lane, e, io.reset_obs, s_o[w][0], s_o[w][1], s_o[w][2], s_o[w][3]);
        }
    }
}

int launch(int dtype, int64_t n, const void *params, const b200env_io *io, uint32_t flags, uint64_t seed, int64_t off,
           const uint8_t *mask, int mode, cudaStream_t s) {
    const P &p = *static_cast<const P *>(params);
    if (p.n_rays < 2 || p.n_rays > B200_UGVO_MAX_RAYS || p.obs_num < 0 || p.obs_num > MAXO) return B200ENV_EPARAMS;
    if (mode == 0) {
        const unsigned grid = (unsigned)((n + G - 1) / G);
        const bool ar = (flags & B200ENV_AUTO_RESET) != 0;
        if (ar && io->work) {
            if (n > (int64_t)0x7fffffff) return B200ENV_ESIZE; // the list holds 32-bit instance indices
            if (cudaMemsetAsync(io->work, 0, sizeof(int32_t), s) != cudaSuccess) return b200_check_launch();
        }
        B200_LAUNCH_TIO(ugvo_step_kernel, grid, TPB, s, p, *io, n, flags, seed, off);
        if (ar) {
            // enough warps to hold every SM at 4 blocks; with the list they stride over it, without it over the batch
            int64_t rgrid = (n + RESET_WARPS * 32 - 1) / (RESET_WARPS * 32);
            if (rgrid > 148 * UGVO_RESET_MINB) rgrid = 148 * UGVO_RESET_MINB;
            B200_LAUNCH_TIO(ugvo_autoreset_kernel, (unsigned)rgrid, RESET_WARPS * 32, s, p, *io, n, seed, off);
        }
    } else {
        const unsigned grid = (unsigned)((n + WARPS - 1) / WARPS);
        B200_LAUNCH_TIO(ugvo_aux_kernel, grid, WARPS * 32, s, p, *io, n, seed, off, mask, mode);
    }
    return b200_check_launch();
}

} // namespace

int ugvo_dims(int variant, int *sf, int *od, int *ad, int *dd) {
    if (variant != 0 && variant != 1) return B200ENV_EENV;
    if (sf) *sf = B200_UGVO_STATE_FIELDS;
    if (od) *od = 4 + B200_UGVO_MAX_RAYS;
    if (ad) *ad = 2;
    if (dd) *dd = 0;
    return B200ENV_OK;
}
int ugvo_step(int dtype, int64_t n, const void *params, const b200env_io *io, uint32_t flags, uint64_t seed, int64_t off,
              cudaStream_t s) {
    if (!io->state || !io->time || !io->action || !io->next_obs || !io->reward || !io->done || !io->flag) return B200ENV_ENULL;
    if ((flags & B200ENV_AUTO_RESET) && !io->episode) return B200ENV_ENULL;
    return launch(dtype, n, params, io, flags, seed, off, nullptr, 0, s);
}
int ugvo_reset(int dtype, int64_t n, const void *params, const b200env_io *io, const uint8_t *mask, uint64_t seed,
               int64_t off, cudaStream_t s) {
    if (!io->state || !io->time || !io->episode) return B200ENV_ENULL;
    return launch(dtype, n, params, io, 0, seed, off, mask, 1, s);
}
int ugvo_observe(int dtype, int64_t n, const void *params, const b200env_io *io, cudaStream_t s) {
    if (!io->state || !io->time || !io->next_obs) return B200ENV_ENULL;
    return launch(dtype, n, params, io, 0, 0, 0, nullptr, 2, s);
}
