/*
 * b200env.h -- C ABI of the B200-native batched environment engine.
 *
 * This is the drop-in boundary for the environment-step hot path of
 * HKPolyU-UAV/ReinforcementLearningPlatform.  The reference has no FFI of its
 * own: its boundary is the duck-typed Python object contract of
 * `algorithm/rl_base.py:4-162` (attributes + reset/step_update/get_state/
 * get_reward/is_Terminal).  Each entry point below names the reference
 * method(s) it replaces; the Python classes in
 * `reinforcementlearningplatform_b200/` re-expose the rl_base attribute names
 * on top of these calls (see INTEGRATION.md).
 *
 * Conventions
 *   - every pointer inside b200env_io is a DEVICE pointer; `params` is a HOST
 *     pointer to one of the POD structs below (copied into kernel-argument
 *     space at launch);
 *   - all per-instance arrays are struct-of-arrays, field-major: element
 *     (field f, instance i) of an array with F fields lives at [f * n + i];
 *   - `dtype` selects the arithmetic/storage type of state, action, dis, obs
 *     and reward (B200ENV_F64 or B200ENV_F32).  `time` is always float64 and
 *     is accumulated with plain IEEE additions exactly as the reference does
 *     (`self.time += h`), so time-out flags are bit-exact in both modes;
 *   - no call blocks: work is enqueued on `stream` (a cudaStream_t, may be 0);
 *   - return value: 0 on success, a negative B200ENV_E* code otherwise.  No
 *     CPU fallback exists: without a CUDA device every launch returns
 *     B200ENV_ECUDA.
 */
#ifndef B200ENV_H
#define B200ENV_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define B200_API __attribute__((visibility("default")))
#else
#define B200_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------ enums */

enum b200env_id {
    B200ENV_CARTPOLE      = 0, /* environment/CartPole/CartPole.py, CartPoleAngleOnly.py (+ PPO2 demo copy) */
    B200ENV_FAS           = 1, /* environment/FlightAttitudeSimulator/FlightAttitudeSimulator.py */
    B200ENV_SOI           = 2, /* environment/SecondOrderIntegration/SecondOrderIntegration.py */
    B200ENV_BALLBALANCER  = 3, /* environment/BallBalancer/BallBalancer1D.py */
    B200ENV_TWOLINK       = 4, /* environment/RobotManipulator/TwoLinkManipulator.py */
    B200ENV_UGV           = 5, /* environment/UGV/UGVForward.py, UGVBidirectional.py */
    B200ENV_UGVO          = 6, /* environment/UGVForwardObstacleAvoidance/UGVForwardObstacleAvoidance.py */
    B200ENV_UAV_ATT       = 7, /* environment/UavFntsmcParam/uav_att_ctrl_RL.py (+ uav.py, FNTSMC.py, ref_cmd.py) */
    B200ENV_UAV_POS       = 8, /* environment/UavFntsmcParam/uav_pos_ctrl_RL.py (+ uav.py, FNTSMC.py, ref_cmd.py) */
    B200ENV_UAVROBUST     = 9, /* environment/UavRobust/Uav{Hover,HoverOuterLoop,InnerLoop,TrackingOuterLoop}.py */
    B200ENV_FAS_DISCRETE  = 10,/* environment/FlightAttitudeSimulator/FlightAttitudeSimulatorDiscrete.py (DQN-family demos) */
    B200ENV_COUNT         = 11
};

enum b200env_dtype { B200ENV_F64 = 0, B200ENV_F32 = 1 };

enum b200env_err {
    B200ENV_OK      =  0,
    B200ENV_EENV    = -1, /* unknown env id / variant */
    B200ENV_EDTYPE  = -2,
    B200ENV_EPARAMS = -3, /* params_bytes does not match the struct of this env */
    B200ENV_ENULL   = -4, /* a required pointer is NULL */
    B200ENV_ECUDA   = -5, /* CUDA error at launch; see b200env_last_cuda_error() */
    B200ENV_ESIZE   = -6  /* n_envs <= 0 or >= 2^31 (one GPU cannot hold more), or a net too wide for K-POLICY */
};

/* step flags */
#define B200ENV_AUTO_RESET 1u /* re-initialise an instance in the same call that sets its `done`
                                 (in-kernel Philox draw with the reference's reset distribution);
                                 replaces the `if env.is_terminal: env.reset(True)` branch of the
                                 train.py loops (e.g. demonstration/PPO2/PPO2-4-CartPoleAngleOnly/train.py:187-191) */

/* ------------------------------------------------------------- I/O bundle */

typedef struct b200env_io {
    void          *state;      /* [state_fields][n]  dtype   persistent per-instance state              */
    double        *time;       /* [n]                f64     `self.time`                                */
    uint32_t      *episode;    /* [n]                u32     episode counter = Philox counter for reset */
    const void    *action;     /* [action_dim][n]    dtype   (step only)                                */
    const void    *dis;        /* [dis_dim][n]       dtype   injected disturbance, may be NULL          */
    void          *obs;        /* [obs_dim][n]       dtype   `current_state` (pre-step obs), may be NULL*/
    void          *next_obs;   /* [obs_dim][n]       dtype   `next_state`  (s' of the transition)       */
    void          *reward;     /* [n]                dtype   `reward`                                   */
    uint8_t       *done;       /* [n]                u8      `is_terminal`                              */
    int32_t       *flag;       /* [n]                i32     `terminal_flag`                            */
    void          *reset_obs;  /* [obs_dim][n]       dtype   obs the policy sees next: s' or, where an
                                                             auto-reset happened, the reset obs; may be NULL */
    int32_t       *work;       /* [1 + n]            i32     optional scratch (may be NULL; contents undefined after
                                                             the call): work[0] counts, work[1..] lists the instances
                                                             that terminated in this step, so that kernels with an
                                                             expensive auto-reset (the obstacle-map rejection sampling
                                                             of B200ENV_UGVO) balance it over the grid */
    int32_t        io_dtype;   /* element type of the RL-facing buffers action, dis, obs, next_obs, reward and
                                  reset_obs: B200ENV_F64 (0) = same as `dtype` (default), B200ENV_F32 = float32 even
                                  when dtype is F64.  The RL side of the reference is float32 (actor output
                                  Proximal_Policy_Optimization2.py:69-76, RolloutBuffer.to_tensor
                                  utils/classes.py:292-301), so float32 I/O with float64 state and arithmetic keeps the
                                  fp64 trajectory and halves the interface bytes (PCIe, rollout buffer). */
    int32_t        pad_;
} b200env_io;

/* Row strides of a time-major rollout (b200env_rollout): row t of an array starts `stride` ELEMENTS (of that array's
 * element type) after row t-1.  For the device-resident buffer of rollout.py: action_stride = action_dim * n,
 * obs_stride = next_obs_stride = obs_dim * n, reward_stride = done_stride = flag_stride = n. */
typedef struct b200env_rollout_spec {
    int64_t steps;
    int64_t action_stride, dis_stride, obs_stride, next_obs_stride, reward_stride, done_stride, flag_stride;
} b200env_rollout_spec;

/* ------------------------------------------------------ per-env parameters */
/* All parameter structs are plain doubles/ints.  The host mirror fills them
 * from the attribute names of the reference classes; thresholds that the
 * reference computes from constants (e.g. `theta_max + deg2rad(1)`) are
 * evaluated on the host with the same expression so comparisons are
 * bit-identical. */

/* CartPole family.  variant 0: CartPole.py (obs 4); 1: CartPoleAngleOnly.py (obs 2, time-loop);
 * 2: demonstration/PPO2/PPO2-4-CartPoleAngleOnly/cartpole_angleonly.py (obs 2, single RK4 step). */
typedef struct b200_cartpole_params {
    double M, m, g, ell, kf;            /* CartPole.py:34-38 */
    double dt, time_max;                /* CartPole.py:41-42 */
    double theta_max, dtheta_max, x_max, dx_max; /* obs normalisers, CartPole.py:26-29 */
    double static_gain;                 /* CartPole.py:31 */
    double norm_boundless;              /* CartPoleAngleOnly.py:28 (dtheta normaliser = 4) */
    double theta_term_hi;               /* theta_max + deg2rad(1)                       CartPole.py:167 */
    double theta_term_lo;               /* -dtheta_max - deg2rad(1) (sic, N2) or -thetaMax - deg2rad(1) */
    double reset_theta_lo, reset_theta_hi; /* U(lo,hi) for theta0, CartPole.py:272 */
    double reset_x_lo, reset_x_hi;         /* U(lo,hi) for x0,     CartPole.py:273 (0,0 for AngleOnly) */
    int32_t variant;
    int32_t pad_;
} b200_cartpole_params;

/* state fields of the CartPole family: theta, dtheta, x, dx */
#define B200_CARTPOLE_STATE_FIELDS 4


/* UavFntsmcParam attitude / position tracking envs (B200ENV_UAV_ATT, B200ENV_UAV_POS).
 * Quadrotor: environment/UavFntsmcParam/uav.py:7-25,93-148; controllers: FNTSMC.py:4-14,47-69,112-137;
 * wrappers: uav_att_ctrl.py, uav_att_ctrl_RL.py, uav_pos_ctrl.py, uav_pos_ctrl_RL.py; references: ref_cmd.py.
 * The per-instance learnable gains, FNTSMC integrators and trajectory parameters live in `state`;
 * everything here is shared by all instances. */
typedef struct b200_uav_params {
    double m, g, J[3], kr, kt;          /* uav.py:9-17 */
    double dt, time_max;                /* uav.py:22-23 (train.py sets 0.02 / 10) */
    double pos_lo[3], pos_hi[3];        /* pos_zone[i][0] - max_admissible_error, pos_zone[i][1] + ...   uav.py:182-193 */
    double att_lo[3], att_hi[3];        /* att_zone[i][0] + deg2rad(1), att_zone[i][1] - deg2rad(1)      uav.py:195-206 */
    double att_zone_min[3], att_zone_max[3]; /* raw zone, used by the att reward penalty uav_att_ctrl_RL.py:96-102 */
    double t_term;                      /* time_max - dt / 2                                             uav.py:216 */
    double init_state[12];              /* concat(pos0, vel0, angle0, pos0) (sic, N5)                    uav.py:64 */
    /* inner-loop (attitude) FNTSMC: fixed in the position env, reset values of the learnable gains in the attitude env */
    double att_k1[3], att_k2[3], att_alpha[3], att_beta[3], att_gamma[3], att_lmd[3];
    /* outer-loop (position) FNTSMC: alpha/beta fixed; k1,k2,gamma,lmd are the reset values of the learnable gains */
    double pos_k1[3], pos_k2[3], pos_alpha[3], pos_beta[3], pos_gamma[3], pos_lmd[3];
    double Q_e[3], Q_de[3], R[3];       /* reward weights: (Q_att,Q_pqr,R) uav_att_ctrl_RL.py:44-46 or (Q_pos,Q_vel,R) uav_pos_ctrl_RL.py:51-53 */
    double ref_amplitude[4], ref_period[4], ref_bias_a[4], ref_bias_phase[4]; /* deterministic trajectory (random_trajectory=False) */
    double dot_att_ref_limit;           /* 60 * pi / 180                                                 uav_pos_ctrl.py:25 */
    double att_limit;                   /* pi / 4                                                        uav_pos_ctrl.py:314 */
    double traj_A_hi[4];                /* random trajectory: A ~ U(0, hi)   uav_att_ctrl.py:157-159 / uav_pos_ctrl.py:405-406 */
    double traj_T_lo, traj_T_hi;        /* random trajectory: T ~ U(lo, hi)  uav_att_ctrl.py:160 / uav_pos_ctrl.py:407 */
    double traj_phase_hi;               /* att: phi0 ~ U(0, pi/2) uav_att_ctrl.py:161; pos: unused (phi0 fixed) */
    double init_pos_r[3];               /* random_pos0: admissible radius r = 0.3 * ones(3)              uav_pos_ctrl.py:512 */
    int32_t random_trajectory;          /* reset_..._tracking(random_trajectory=...) */
    int32_t yaw_fixed;
    int32_t random_pos0;                /* position env, layout variant 1 only: reset_uav_pos_ctrl(random_pos0=True) */
    int32_t pad_;
} b200_uav_params;

/* The `state` buffer of B200ENV_UAV_ATT, B200ENV_UAV_POS and B200ENV_UAVROBUST is BLOCK-INTERLEAVED, not field-major: instances are grouped in
 * blocks of 128, every block holds B200_UAV_STATE_SLOTS field slots of 128 values, element (field f, instance i) lives at
 * [((i / 128) * B200_UAV_STATE_SLOTS + f) * 128 + i % 128], and the buffer has b200env_state_elems() elements (n rounded up to
 * a multiple of 128).  The kernels then reach every field of an instance with one base register plus an immediate offset
 * (11 % faster than [field][n] for the position env, whose step touches 66 state fields).  Callers that only hand the buffer
 * back never notice; callers that inject or read states use the formula (b200env_state_layout reports block and slots; the
 * Python mirror converts in get_state_buffers / set_state_buffers).  All other buffers, and `state` of every other env, stay
 * field-major. */
#define B200_UAV_STATE_BLOCK 128
#define B200_UAV_STATE_SLOTS 64
/* state fields, attitude env: phi theta psi p q r | s1[3] | k1[3] k2[3] gamma[3] lmd[3] | A[3] T[3] phase[3] | ref[3] dot_ref[3] */
#define B200_UAV_ATT_STATE_FIELDS 36
/* state fields, position env: x y z vx vy vz phi theta psi p q r | sigma_o1[3] | s1[3] | att_ref[3] |
 *                             k1[3] k2[3] gamma[3] lmd[3] | A[4] T[4] phase[4] | pos_ref[3] dot_pos_ref[3] */
#define B200_UAV_POS_STATE_FIELDS 51
/* Layout variant 1 of the position env (b200env_dims(B200ENV_UAV_POS, 1)) appends next_pqr0[3], the reference's
 * `init_state[9:12]`: with random_pos0=True every reset draws pos0 ~ U(trajectory[0] - r, trajectory[0] + r)
 * (set_random_init_pos, uav_pos_ctrl.py:457-465,510-513) and, because init_state = concat(pos0, vel0, angle0, pos0)
 * (uav.py:268, note N5), loads p, q, r from the pos0 of the PREVIOUS reset.  Reproduced as is; the three fields are
 * only touched by resets. */
#define B200_UAV_POS_STATE_FIELDS_V1 54
/* `ref/dot_ref` (att) and `pos_ref/dot_pos_ref` (pos) are only stored on a terminal step without auto-reset and read by
 * b200env_reset / b200env_observe: the reference's reset does not clear them, so the first observation of the next
 * episode is taken against the previous episode's last reference (uav_att_ctrl.py:187-216, uav_pos_ctrl.py:488-533). */

/* Flight_Attitude_Simulator (B200ENV_FAS): environment/FlightAttitudeSimulator/FlightAttitudeSimulator.py:9-287;
 * PPO2/DPPO2 demo copy = same code with timeMax = 10, Q = 1, R = 0.05 (flight_attitude_simulator.py:42,211-224). */
typedef struct b200_fas_params {
    double L, k, mgd, denom;            /* L; k; m*g*dis; J + m*dis**2          :232-236 (host-evaluated) */
    double dt, time_max;                /* :38, :42 */
    double min_theta, max_theta, min_omega, max_omega, static_gain; /* obs normalisation :173-185 */
    double theta_term_hi, theta_term_lo; /* maxTheta + deg2rad(1), minTheta - deg2rad(1)   :199-206 */
    double Q, R;                        /* reward weights :218-219 */
    double reset_lo, reset_hi;          /* theta0 ~ U(minTheta, maxTheta) :270-271 */
} b200_fas_params;
#define B200_FAS_STATE_FIELDS 2         /* theta, dTheta */

/* FlightAttitudeSimulatorDiscrete (B200ENV_FAS_DISCRETE): environment/FlightAttitudeSimulator/
 * FlightAttitudeSimulatorDiscrete.py:9-274.  The action is the force VALUE picked from the discrete action_space
 * (:56-59); the dynamics are the file's own closure f() (:199-203, incl. its `dis + m dis^2` denominator) integrated by
 * `while t_sim <= dt` with h = dt, i.e. TWO RK4 steps of h = dt per control period (:205-219), followed by the
 * +-theta_max bounce (:220-225). */
typedef struct b200_fas_discrete_params {
    double a2, a1;                      /* -k/(J+m d^2); -m g d/(d + m d^2) (sic)          :202-203 (host-evaluated) */
    double L, denom;                    /* a0 = L * action / (J + m d^2)                   :204 */
    double dt, time_max;                /* :28, :30 */
    double theta_max, dtheta_max, static_gain; /* :23-25 */
    double theta_out;                   /* theta_max + deg2rad(1)                          :170-177 */
    double Q, R;                        /* get_reward locals :233-234 */
    double bounce;                      /* -0.8                                            :222,225 */
} b200_fas_discrete_params;
#define B200_FAS_DISCRETE_STATE_FIELDS 2 /* theta, dTheta */

/* SecondOrderIntegration (B200ENV_SOI): environment/SecondOrderIntegration/SecondOrderIntegration.py:13-352;
 * DPPO2 demo copy: obs multiplied by static_gain, success terminal disabled, Q_vel = Q_acc = 0. */
typedef struct b200_soi_params {
    double map_x, map_y, target_x, target_y; /* :16-17 */
    double mass, k, vmax, dt, time_max, admissible_error; /* :31-42 */
    double obs_gain;                    /* 1 (ENV) or static_gain (DPPO2 copy :213) */
    double Q_pos, Q_vel, Q_acc;         /* :262-264 */
    double reset_margin;                /* pos0 ~ U(0 + 0.1, map - 0.1) :329-331 */
    int32_t success_terminal;           /* 1 (ENV :246-249) / 0 (DPPO2 copy) */
    int32_t pad_;
} b200_soi_params;
#define B200_SOI_STATE_FIELDS 4         /* x, y, vx, vy */

/* BallBalancer1D (B200ENV_BALLBALANCER): environment/BallBalancer/BallBalancer1D.py:14-322 */
typedef struct b200_ballbalancer_params {
    double K, L;                        /* :62-63, :58 */
    double omega_min, omega_max, theta_min, theta_max, v_min, v_max; /* :34-39 */
    double dt, time_max, static_gain, target; /* :47-51, :70 */
    double deg1;                        /* deg2rad(1) :214 */
    double reset_theta_lo, reset_theta_hi, reset_pos_lo, reset_pos_hi, init_vel; /* :294-296 */
} b200_ballbalancer_params;
#define B200_BALLBALANCER_STATE_FIELDS 4 /* pos, vel, theta, error (error lags one step inside is_Terminal, :279-281) */

/* TwoLinkManipulator (B200ENV_TWOLINK): environment/RobotManipulator/TwoLinkManipulator.py:8-312 */
typedef struct b200_twolink_params {
    double l, m, g, J;                  /* :33-36 */
    double dt, time_max;                /* :37-39 */
    double base_x, base_y;              /* :32 */
    double theta_max, miss, omega_ok;   /* pi; 0.01; deg2rad(5)  :42-48,194-197 */
    double init_end_x, init_end_y;      /* init_endPos :19 (error after reset = target - init_endPos, :300) */
    double r2_lo, r2_hi;                /* target radius^2 ~ U(0.3^2, (2l)^2) :286 */
    double Q_pos, Q_omega, Q_acc;       /* :212-214 */
} b200_twolink_params;
#define B200_TWOLINK_STATE_FIELDS 8     /* theta1 theta2 omega1 omega2 err_x err_y target_x target_y */

/* UGVForward / UGVBidirectional (B200ENV_UGV): environment/UGV/UGVForward.py:10-362, UGVBidirectional.py:10-367 */
typedef struct b200_ugv_params {
    double map_x, map_y, target_x, target_y;
    double dt, time_max, kf, kt;        /* :43-48 */
    double e_max, v_max, e_phi_max, omega_max, static_gain; /* :53-58,66 */
    double Q_pos, Q_vel, Q_phi, Q_omega; /* :264-267 */
    double reset_d0;                    /* pos0 ~ U(d0, map - d0) :336-338 */
    int32_t bidirectional;              /* 0 UGVForward, 1 UGVBidirectional */
    int32_t pad_;
} b200_ugv_params;
#define B200_UGV_STATE_FIELDS 5         /* x, y, vel, phi, omega */

/* UGVForwardObstacleAvoidance (B200ENV_UGVO): environment/UGVForwardObstacleAvoidance/UGVForwardObstacleAvoidance.py:11-557
 * + map.py:65-80,120-174.  variant 0 = that file; variant 1 = the PPO2/DPPO2 demo copies
 * (demonstration/DPPO2/DPPO2-4-UGVForwardObstacleAvoidance/UGVForwardObstacleAvoidance.py: dt = 0.05, progress reward
 * :449-473, is_success ignores omega :421-427, rk44 freezes the pose when the PREVIOUS vel < 0 :488-509). */
typedef struct b200_ugvo_params {
    double map_x, map_y;
    double dt, time_max, kf, kt;                 /* :42-47 */
    double e_max, v_max, e_phi_max, omega_max, static_gain; /* :58-63,71 */
    double r_vehicle;                            /* :38 */
    double laser_dis, laser_blind, laser_range;  /* :49-51 */
    double Q_pos, Q_vel, Q_phi, Q_omega;         /* :452-455 (variant 0) */
    double safety_dis_obs, safety_dis_st, r_min, r_max, st_margin; /* reset: :529-537, map.py:67 */
    int32_t n_rays;                              /* laserState = int(2 * range / step) + 1 = 37   :53 */
    int32_t obs_num;                             /* obstacles drawn at reset (10 ENV/PPO2, 15 DPPO2), <= B200_UGVO_MAX_OBS */
    int32_t variant;
    int32_t pad_;
} b200_ugvo_params;
#define B200_UGVO_MAX_OBS 16
#define B200_UGVO_MAX_RAYS 37
/* state fields: x y vel phi omega | target_x target_y | n_obs | (cx, cy, r) x B200_UGVO_MAX_OBS */
#define B200_UGVO_STATE_FIELDS (8 + 3 * B200_UGVO_MAX_OBS)
/* Reset draws (Philox4x32-10 block index = counter word 3; two doubles per block):
 *   block 0: start;  blocks 1..64: target candidates (first with |t - s| >= safety_dis_st);  block 100: phi0;
 *   obstacle k, candidate c: blocks 1000 + 2 * (2048 k + c) (centre) and + 1 (radius).  Candidates are tried in index
 *   order, at most 2048 per obstacle (the reference retries without bound, map.py:171-172); if none is legal the map
 *   keeps the obstacles placed so far. */

/* UavRobust (B200ENV_UAVROBUST): the same quadrotor (environment/UavRobust/uav.py:429-560) wrapped as four RL envs.
 * variant 0 uav_hover_outer_loop   UavHoverOuterLoop.py:81-196    obs 6, action = virtual acceleration (3), inner loop by FNTSMC
 * variant 1 uav_hover              UavHover.py:101-226            obs 12, action = acceleration (3) + torque (3)
 * variant 2 uav_inner_loop         UavInnerLoop.py:88-210         obs 6, action = torque (3), attitude only
 * variant 3 uav_tracking_outer_loop UavTrackingOuterLoop.py:90-255 obs 6, action = virtual acceleration (3), sinusoidal reference
 * Inner-loop FNTSMC with torque saturation: UavRobust/FNTSMC.py:80-106. */
typedef struct b200_uavrobust_params {
    double m, g, J[3], kr, kt;
    double dt, time_max, t_term;            /* t_term = time_max - dt / 2                   uav.py:545 */
    double pos_zone_min[3], pos_zone_max[3];/* no margins here                              uav.py:511-525 */
    double att_zone_min[3], att_zone_max[3];/*                                              uav.py:527-541 */
    double pos0[3], vel0[3], angle0[3], pqr0[3]; /* reset state (here pqr0 IS used)         UavHover.py:178-189 */
    double att_k1[3], att_k2[3], att_alpha[3], att_beta[3], att_gamma[3], att_lmd[3], att_saturation[3];
    double e_pos_span[3];                   /* e_pos_max - e_pos_min                        UavHover.py:38-39 */
    double vel_span[3];                     /* vel_max - vel_min  (e_vel_max - e_vel_min)   UavHover.py:40-41 */
    double e_att_span[3];                   /* e_att_max - e_att_min                        UavHover.py:47-48 */
    double e_dot_att_span_neg[3];           /* e_dot_att_min - e_dot_att_max  (sic, N10)    UavHover.py:109, UavInnerLoop.py:94 */
    double dot_att_min[3], dot_att_max[3];  /* reference-rate limits                        UavHover.py:42-43 */
    double static_gain;
    double Qx, Qv, R;                       /* reward weights (get_reward locals) */
    double ref_bias_a[3];                   /* tracking: centre of pos_zone; inner loop: zeros */
    double target_lo[3], target_hi[3];      /* hover: pos_ref ~ U(zone_min + 1, zone_max - 1)   UavHover.py:224-226 */
    double sig_A_hi[3];                     /* random reference amplitude upper bounds (variants 2, 3) */
    double sig_T_lo, sig_T_hi, sig_phase_hi;/* U(3,6) / U(5,10); U(0, pi/2) */
    double init_pos_r;                      /* tracking: initial position within +-0.3 of the trajectory start */
    int32_t variant;
    int32_t pad_;
} b200_uavrobust_params;
/* state fields: x y z vx vy vz phi theta psi p q r | s1[3] | att_ref[3] | dot_att_ref[3] | pos_ref[3] | A[3] T[3] phase[3] */
#define B200_UAVROBUST_STATE_FIELDS 33

/* ---------------------------------------------------------------- queries */

/* sizes of the SoA arrays of one env family/variant; any out pointer may be NULL */
B200_API int b200env_dims(int env_id, int variant, int *state_fields, int *obs_dim, int *action_dim, int *dis_dim);

/* sizeof() of the params struct the library was compiled with (ABI check) */
B200_API size_t b200env_params_bytes(int env_id);

/* last cudaError_t seen by a failed launch in this thread (0 if none) */
B200_API int b200env_last_cuda_error(void);
B200_API const char *b200env_version(void);

/* ------------------------------------------------------------- hot path */

/* One control period for n instances: replaces `env.step_update(action)` of every
 * environment (algorithm/rl_base.py:126; e.g. CartPole.py:257-264) -- obs = get_state(),
 * rk44(action), is_Terminal(), next_obs = get_state(), get_reward() -- and, with
 * B200ENV_AUTO_RESET, the following `env.reset(True)`.
 * For the UavFntsmcParam envs the default action is the 8 controller gains and the call
 * fuses `get_param_from_actor(a)` + `generate_action_4_uav()`/`att_control()` +
 * `step_update()` (train.py:292-297 of PPO2-4-UavFntsmcParamPos). */
B200_API int b200env_step(int env_id, int dtype, int64_t n_envs,
                 const void *params, size_t params_bytes,
                 const b200env_io *io, uint32_t flags,
                 uint64_t seed, int64_t env_index_offset, void *cuda_stream);

/* Replaces `env.reset(random=True)` (rl_base.py:161; e.g. CartPole.py:266-295) for the
 * instances whose mask byte is non-zero (mask == NULL: all).  Draws the reference's
 * reset distribution from Philox4x32-10 keyed by (seed, env_index_offset + i, episode[i]),
 * increments episode[i], zeroes time[i] and writes the initial observation to
 * io->next_obs (if not NULL). */
B200_API int b200env_reset(int env_id, int dtype, int64_t n_envs,
                  const void *params, size_t params_bytes,
                  const b200env_io *io, const uint8_t *mask,
                  uint64_t seed, int64_t env_index_offset, void *cuda_stream);

/* Replaces `env.get_state()` (rl_base.py:158): observation of the current state into
 * io->next_obs without stepping.  Used after the caller injected a state. */
B200_API int b200env_observe(int env_id, int dtype, int64_t n_envs,
                    const void *params, size_t params_bytes,
                    const b200env_io *io, void *cuda_stream);

/* ------------------------------------------------------------- GAE */

/* Replaces the reverse loop of Proximal_Policy_Optimization2.learn (algorithm/policy_base/
 * Proximal_Policy_Optimization2.py:88-98) and Worker.learn (Distributed_PPO2.py:59-69) for N env columns at once.
 * All arrays are device float32, time-major [T][N] (element (t, n) at t * N + n); `done`/`success` hold 0.0/1.0 like
 * the reference's RolloutBuffer (utils/classes.py:250-301).
 *   delta = r + gamma * (1 - success) * vs_next - vs;  gae_t = delta_t + gamma * lmd * gae_{t+1} * (1 - done_t)
 *   adv = gae;  v_target = adv + vs
 * acc_mode 0: float32 sequential, bit-identical to the reference loop under numpy >= 2; 1: float64 carry (numpy 1.x);
 * 2: the float64-carry scan evaluated as a warp-level parallel scan along time (one warp per column, 32 time steps per
 *    trip composed by shuffles): for rollouts with few columns -- the reference's own shape is N = 1 -- where one thread
 *    per column leaves the GPU empty; equal to mode 1 up to float64 reassociation (<= 1 float32 ulp in the outputs).
 * stats (device double[3], may be NULL) is INCREMENTED by (sum adv, sum adv^2, T * N): zero it first; all-reduce it
 * over ranks for a global advantage normalisation.  scratch (device, 8-byte aligned, b200_gae_scratch_bytes(N) bytes,
 * may be NULL): with it the sums are reduced in a fixed order -- the same bits on every run; without it the per-block
 * partial sums are added atomically (order-dependent in the last bits). */
B200_API size_t b200_gae_scratch_bytes(int64_t N);
B200_API int b200_gae(int64_t T, int64_t N, const float *r, const float *vs, const float *vs_next, const float *done,
                      const float *success, double gamma, double lmd, int acc_mode, float *adv, float *v_target,
                      double *stats, void *scratch, size_t scratch_bytes, void *cuda_stream);

/* Layout of the persistent `state` buffer of an env family: *block = 0 -> field-major [state_fields][n_envs]; *block = B > 0
 * -> block-interleaved with *slots field slots per block of B instances (the UAV families, see B200_UAV_STATE_SLOTS above).
 * b200env_state_elems: number of elements the caller must allocate for n_envs instances. */
B200_API int b200env_state_layout(int env_id, int variant, int *block, int *slots);
B200_API size_t b200env_state_elems(int env_id, int variant, int64_t n_envs);

/* `spec->steps` control periods with pre-computed actions in one call: the collection loop of the train scripts
 * (`while buffer_index < batch_size: step_update; buffer.append`, PPO2-4-CartPoleAngleOnly/train.py:186-216) when the
 * actions do not depend on the observations (random-action benchmarks, open-loop replays) or are produced on the
 * device ahead of time.  io->action / dis / obs / next_obs / reward / done / flag point at row 0 of time-major arrays
 * whose rows are `spec` strides apart; reset_obs receives the observation after the last step.  Families built on the
 * generic one-thread-per-instance kernel (FAS, SOI, BallBalancer, TwoLink, UGV) run all steps in ONE launch with the
 * instance state held in registers; the others launch their step kernel once per time step. */
B200_API int b200env_rollout(int env_id, int dtype, int64_t n_envs, const void *params, size_t params_bytes,
                             const b200env_io *io, const b200env_rollout_spec *spec, uint32_t flags, uint64_t seed,
                             int64_t env_index_offset, void *cuda_stream);

/* Same scan over a device-resident rollout as the step kernels write it (rollout.py): `done` is the u8 is_terminal
 * column, `flag` the i32 terminal_flag column, and success = done && flag != timeout_flag -- the rule by which the
 * train loops fill RolloutBuffer.success (demonstration/PPO2/PPO2-4-CartPoleAngleOnly/train.py:198-205,
 * PPO2-4-UavFntsmcParamPos/train.py:299-302).  25 instead of 28 bytes of HBM traffic per element. */
B200_API int b200_gae_flags(int64_t T, int64_t N, const float *r, const float *vs, const float *vs_next,
                            const uint8_t *done, const int32_t *flag, int32_t timeout_flag, double gamma, double lmd,
                            int acc_mode, float *adv, float *v_target, double *stats, void *scratch,
                            size_t scratch_bytes, void *cuda_stream);

/* adv <- (adv - mean) / (std + eps) with the unbiased std (torch.Tensor.std) derived from stats = (sum, sum of
 * squares, count): Proximal_Policy_Optimization2.py:99-100 (eps = 1e-5); a true float32 division per element. */
B200_API int b200_adv_normalize(int64_t count, float *adv, const double *stats, double eps, void *cuda_stream);

/* Monte-Carlo return scan of PPO / DPPO (v1): algorithm/policy_base/Proximal_Policy_Optimization.py:113-119,
 * Distributed_PPO.py:58-64.  r is [T][N] in r_dtype (B200ENV_F64 like RolloutBuffer.r, or B200ENV_F32), done [T][N] u8;
 * the recurrence `R = 0 if done; R = r + gamma * R` runs backwards in float64, returns [T][N] are float32 like
 * `torch.tensor(np.array(rewards), dtype=torch.float32)`. */
B200_API int b200_mc_returns(int r_dtype, int64_t T, int64_t N, const void *r, const uint8_t *done, double gamma,
                             float *returns, void *cuda_stream);

/* The same scan (returns bit-identical to b200_mc_returns) that also INCREMENTS stats (device double[3]) by
 * (sum R, sum R^2, T * N) over the stored float32 returns, summed in float64: the statistics b200_adv_normalize reads,
 * for the v1 return normalisation R_hat = (R - mean) / (std + eps); all-reduce them over ranks first for a global one.
 * The sums are reduced in a fixed order through scratch (device, 8-byte aligned, b200_gae_scratch_bytes(N) bytes): the
 * same bits on every run.  Errors, all returned before any CUDA call: B200ENV_ESIZE (T <= 0, N <= 0 or N >= 2^31),
 * B200ENV_EDTYPE (r_dtype), B200ENV_ENULL (r, done, returns, stats or scratch NULL), B200ENV_EPARAMS (scratch too small
 * or misaligned). */
B200_API int b200_mc_returns_stats(int r_dtype, int64_t T, int64_t N, const void *r, const uint8_t *done, double gamma,
                                   float *returns, double *stats, void *scratch, size_t scratch_bytes, void *cuda_stream);

/* K-EPISODE: episode returns, lengths and end reasons of an auto-reset rollout -- the per-episode reward sums of the
 * reference's train loops and their deterministic test episodes, for N instance columns at once.  r is [T][N] in r_dtype
 * (B200ENV_F32 / B200ENV_F64), done [T][N] u8 and flag [T][N] i32: the rollout columns the step kernels write (with T = 1
 * an env's own reward / is_terminal / terminal_flag buffers).  Every done row ends an episode, so the rollout must come
 * from an env stepped with B200ENV_AUTO_RESET.
 * Per instance n, for t = 0 .. T-1:  acc_return[n] = acc_return[n] + (double)r[t][n] (one rounded float64 add);
 *   acc_length[n] += 1;  if done[t][n]: emit (acc_return[n], acc_length[n], flag[t][n]) and zero the carry.
 * acc_return (f64 [N]) and acc_length (i32 [N]) are the caller-owned carry of the episode in progress; zero them when
 * the env is reset.  ep_return (f64), ep_length, ep_flag (i32), each [N] and each may be NULL: the last episode emitted
 * by instance n (left untouched if it emitted none).  first_only = 1: an instance whose ep_flag is not -1 emits nothing
 * (each instance contributes its first episode only; needs ep_flag, initialised to -1 by the caller).
 * stats (device double[B200_EPISODE_STATS], may be NULL) is INCREMENTED over the emitted episodes:
 *   [0] count  [1] sum return  [2] sum return^2  [3] sum length  [4] sum length^2
 *   [5 + f] episodes that ended with flag f, f = 0 .. 15  [21] episodes with any other flag
 * so it can be summed over calls and all-reduced over ranks.  It needs scratch (device, 8-byte aligned,
 * b200_episode_scratch_bytes(N) bytes): per-block partials added in a fixed order, the same bits on every run.
 * Errors, all returned before any CUDA call: B200ENV_ESIZE (T <= 0, N <= 0 or N >= 2^31), B200ENV_EDTYPE (r_dtype),
 * B200ENV_ENULL (r, done, flag or the carry NULL; ep_flag NULL with first_only; scratch NULL with stats),
 * B200ENV_EPARAMS (scratch too small or misaligned). */
#define B200_EPISODE_STATS 22
B200_API size_t b200_episode_scratch_bytes(int64_t N);
B200_API int b200_episode_scan(int r_dtype, int64_t T, int64_t N, const void *r, const uint8_t *done,
                               const int32_t *flag, double *acc_return, int32_t *acc_length, double *ep_return,
                               int32_t *ep_length, int32_t *ep_flag, int first_only, double *stats, void *scratch,
                               size_t scratch_bytes, void *cuda_stream);

/* ------------------------------------------------------------- running normalisation */

/* Replaces RunningMeanStd.update + Normalization.__call__ (utils/classes.py:626-656) as used on rewards
 * (demonstration/PPO2/PPO2-4-CartPoleAngleOnly/train.py:139,210) and UAV observations
 * (PPO2-4-UavFntsmcParamPos/train.py:291,308).  Running state: double run[3][dim] = (n, mean, S); the reference's
 * `std` is n == 1 ? mean (sic, `self.std = x`) : sqrt(S / n).  x, y: [dim][n] field-major in `dtype`.
 *
 * b200_norm_seq: the reference recurrence sample by sample over `rows` samples (x, y = [dim][rows]); bit-exact.
 *   y may be NULL (update only); update = 0 normalises with the stored statistics.
 * b200_norm_batch_stats: (count, mean, M2) of one batch of n instances per feature -> batch_stats[3][dim], summed in
 *   float64 about run's mean (run may be NULL).  scratch: b200_norm_scratch_bytes(dim) bytes, zeroed once by the caller.
 * b200_norm_merge_apply: merges n_batches batch statistics (batch_stats[n_batches][3][dim], e.g. all-gathered over
 *   ranks, merged in index order) into run_in -> run_out (may alias only if y == NULL), then y = (x - mean) / (std +
 *   eps) with the MERGED statistics (y may be x: in-place normalisation).  The merge is Chan's pairwise update written so that a batch of one sample is
 *   bit-identical to the reference's update; update = 0 skips the merge (evaluation: `update=False`).
 * b200_norm_rows_prefix: a whole rollout of ONE scalar feature (the reward column, `r = reward_norm(env.reward)` of
 *   PPO2-4-CartPoleAngleOnly/train.py:210 applied T times) in three launches instead of 2 T: (1) b200_norm_batch_stats with
 *   dim = rows over the time-major [rows][n] buffer gives every row's batch statistics, (2) this call merges them row after
 *   row into the running (n, mean, S) -- batch_stats[n_batches][3][rows], each row's batches in index order -- and stores the
 *   state after every row in cum[3][rows] and the final one in run_out[3], (3) b200_norm_merge_apply with dim = rows,
 *   run_in = cum and update = 0 normalises row t with the statistics after rows 0..t, as the per-row calls would. */
B200_API size_t b200_norm_scratch_bytes(int dim);
B200_API int b200_norm_seq(int dtype, int64_t rows, int dim, const void *x, void *y, double *run, int update, double eps,
                           void *cuda_stream);
B200_API int b200_norm_batch_stats(int dtype, int64_t n, int dim, const void *x, const double *run, double *batch_stats,
                                   void *scratch, void *cuda_stream);
B200_API int b200_norm_merge_apply(int dtype, int64_t n, int dim, const void *x, void *y, const double *batch_stats,
                                   int n_batches, const double *run_in, double *run_out, int update, double eps,
                                   void *cuda_stream);
B200_API int b200_norm_rows_prefix(int rows, const double *batch_stats, int n_batches, const double *run_in, double *cum,
                                   double *run_out, void *cuda_stream);

/* ------------------------------------------------------------- batched policy forward */

/* A small tanh MLP as torch.nn.Linear stores it: layer l maps dims[l] -> dims[l + 1]; w[l] is the DEVICE pointer of
 * `weight` ([dims[l+1]][dims[l]] row-major, float32), b[l] of `bias`.  Hidden layers use tanh; out_act selects the
 * output activation: 0 identity (PPOCritic.forward, utils/classes.py:610-614), 1 relu (PPOActor_Gaussian.forward
 * :563-569). */
typedef struct b200_mlp {
    int32_t n_layers;       /* 1..4 */
    int32_t dims[5];
    int32_t out_act;        /* 0 identity, 1 relu, 2 tanh mapped onto [a_min, a_max] (actor heads of the DPPO2 demos) */
    int32_t pad_;
    const float *w[4];
    const float *b[4];
} b200_mlp;

/* Replaces Proximal_Policy_Optimization2.choose_action (algorithm/policy_base/Proximal_Policy_Optimization2.py:69-76)
 * and the critic forward of learn() (:88-90) for n instances: obs [S][n] float32 field-major (the step kernels'
 * policy-state buffer) ->  mean = actor(obs);  action = clamp(mean + std * eps, a_min, a_max);
 * log_prob = Normal(mean, std).log_prob(action);  value = critic(obs).  eps = noise[A][n] if given, else N(0,1) from
 * Philox4x32-10 keyed by (seed, env_index_offset + i, step) (Box-Muller).  actor or critic may be NULL (then action /
 * value are not written); log_prob, mean may be NULL.  a_min, a_max: device float32 [A].  All nets must fit in shared
 * memory together with the tile's activations (the reference's 64-64-32 / 64-32 nets use ~110 KB) and no layer may be
 * wider than 64, else B200ENV_ESIZE. */
/* precision: must be B200_POLICY_FP32 = float32 FMA pipe, sums in k order (<= 2e-6 absolute from torch's float32 GEMM);
 * any other value returns B200ENV_EPARAMS before any CUDA call.  This kernel keeps every net in shared memory and
 * rejects layers wider than 64 (B200ENV_ESIZE); the tcgen05 path below has neither limit and is the one the Python
 * mirror uses by default. */
#define B200_POLICY_FP32   0
B200_API int b200_policy_forward(int64_t n, const b200_mlp *actor, const b200_mlp *critic, const float *obs,
                                 const float *a_min, const float *a_max, float std, const float *noise, uint64_t seed,
                                 uint64_t step, int64_t env_index_offset, int precision, float *action,
                                 float *log_prob, float *mean, float *value, void *cuda_stream);

/* The same forward on the 5th-generation tensor cores (tcgen05.mma, accumulators in TMEM, weights fed by bulk-copy TMA;
 * csrc/policy_umma.cu): 128-instance tiles, 3xTF32 split (<= 5e-6 absolute on the reference's 64-wide nets, <= 2e-5 on
 * 256-wide ones whose fp32 sums are 4x longer), layers up to 256 wide -- the 41-256-256-{2,1} nets of
 * demonstration/DPPO2/DPPO2-4-UGVForwardObstacleAvoidance/train.py:26-107.  The weights are first packed into a
 * caller-owned device workspace (128-byte aligned, b200_policy_workspace_bytes) in the tensor core's operand layout:
 * b200_policy_pack once per optimizer step, b200_policy_forward_packed once per env step (it reads only dims / out_act
 * from the two structs).  actor->out_act = 2 selects the range-mapped head of those demo nets, mean = tanh(z) * gain + off
 * with off = (a_min + a_max) / 2, gain = a_max - off; std_vec (device float32 [A], may be NULL -> scalar std) is their
 * per-dimension init_std.  Output heads: <= 16 actions, critic 1. */
B200_API size_t b200_policy_workspace_bytes(const b200_mlp *actor, const b200_mlp *critic);
B200_API int b200_policy_pack(const b200_mlp *actor, const b200_mlp *critic, void *workspace, size_t workspace_bytes,
                              void *cuda_stream);
B200_API int b200_policy_forward_packed(int64_t n, const b200_mlp *actor, const b200_mlp *critic, const void *workspace,
                                        size_t workspace_bytes, const float *obs, const float *a_min, const float *a_max,
                                        float std, const float *std_vec, const float *noise, uint64_t seed, uint64_t step,
                                        int64_t env_index_offset, float *action, float *log_prob, float *mean,
                                        float *value, void *cuda_stream);

/* ------------------------------------------------------------- PPO2 / DPPO2 update (K-LEARN) */

/* One mini-batch of the update loop of Proximal_Policy_Optimization2.learn (algorithm/policy_base/
 * Proximal_Policy_Optimization2.py:102-131; the DPPO2 worker copies Distributed_PPO2.py:77-104) taken straight from the
 * device-resident rollout (rollout.py: time-major, field-major float32):  s [T][S][N], a [T][A][N], a_lp [T][A][N]
 * (per-dimension log-probabilities at collection time), adv [T][N] (already normalised), v_target [T][N].  Sample
 * b = t * N + i.  The mini-batch is positions first .. first + count - 1 of
 *   - `index` (device int64 [>= first + count], values in [0, T * N)) when given -- a caller-made permutation;
 *   - else of the pseudo-random permutation of [0, T * N) keyed by `perm_key` (a 6-round Feistel network with cycle
 *     walking, evaluated per sample inside the kernel: the BatchSampler(SubsetRandomSampler(range(B)), mb, False) of
 *     PPO2.py:104 without materialising the permutation; one key per epoch visits every sample exactly once). */
typedef struct b200_ppo2_batch {
    int64_t T, N;
    const float *s, *a, *a_lp, *adv, *v_target;
    const int64_t *index;
    int64_t first, count;
    uint64_t perm_key;
} b200_ppo2_batch;

/* b200_ppo2_grad: forward, loss, backward of BOTH nets for one mini-batch in one launch (fp32 FMA pipe, register-tiled
 * GEMMs over 128-sample tiles held in shared memory; weights resident in shared memory):
 *   actor  (PPO2.py:106-117):  mean = head(actor(s));  lp = sum_d Normal(mean_d, std_d).log_prob(a_d);
 *          ratio = exp(lp - sum_d a_lp_d);  loss = mean(-min(ratio * adv, clamp(ratio, 1 - eps_clip, 1 + eps_clip) * adv))
 *          (the entropy bonus of a fixed-std Gaussian is a constant: it shifts the loss value by -entropy_coef * H and
 *          has no gradient; loss_out[0] includes it);
 *   critic (PPO2.py:123-124):  loss = mse(v_target, critic(s)).
 * Gradients of the MEAN losses with respect to every weight and bias are written to grad_actor / grad_critic (device
 * float32, in torch's parameter order: per layer `weight` [out][in] row-major, then `bias`), summed over samples in a
 * fixed order (per-block partial sums in `workspace`, added up in block order by a second small launch: bit-reproducible
 * for a given device).
 * loss_out: device float32 [2] = (actor loss, critic loss).  Either net may be NULL.  std_vec (device [A]) overrides
 * the scalar std.  a_min / a_max are only read for actor->out_act == 2.
 * Limits of this kernel: every layer <= 64 wide, state_dim <= 64, <= 16 actions, <= 4 layers per net (the nets of
 * every PPO2 demo, utils/classes.py:529-615); wider nets return B200ENV_ESIZE.
 * workspace: b200_ppo2_workspace_bytes() bytes of device memory (contents irrelevant). */
B200_API size_t b200_ppo2_workspace_bytes(const b200_mlp *actor, const b200_mlp *critic);
B200_API int b200_ppo2_grad(const b200_ppo2_batch *batch, const b200_mlp *actor, const b200_mlp *critic, float std,
                            const float *std_vec, const float *a_min, const float *a_max, float eps_clip,
                            float entropy_coef, float *grad_actor, float *grad_critic, float *loss_out, void *workspace,
                            size_t workspace_bytes, void *cuda_stream);

/* The gradient of one PPO v1 update (the v1 demos' joint loss, restated):
 *   V = critic(s);  adv = R_hat - V (no gradient through adv);  ratio and the clipped surrogate as b200_ppo2_grad;
 *   loss = mean(-min(ratio adv, clamp(ratio, 1 - eps_clip, 1 + eps_clip) adv)) + value_coef mse(V, R_hat) - entropy_coef H
 * batch->v_target holds R_hat (the normalised returns) and batch->adv is a caller-owned [T][N] buffer that this call
 * WRITES at the batch's samples (one float32 subtraction R_hat - V); value (device [T][N], may be NULL) receives V there.
 * Three launches: the critic forward over the batch (V bit-identical to the V of b200_ppo2_grad's critic), the
 * b200_ppo2_grad kernel, and its reduction with the critic's gradient and loss multiplied by value_coef: grad_critic is
 * value_coef times b200_ppo2_grad's critic gradient for v_target = R_hat, bit for bit, and loss_out[1] = value_coef mse.
 * Both nets are required.  Errors, all returned before any CUDA call: B200ENV_ENULL (batch, actor, critic or a pointer
 * b200_ppo2_grad needs), B200ENV_EPARAMS (value_coef < 0 or NaN; adv or value overlapping each other or an input:
 * v_target, s, a, a_lp, index; and b200_ppo2_grad's), B200ENV_ESIZE (as b200_ppo2_grad).  workspace: b200_ppo2_workspace_bytes(actor, critic) bytes. */
B200_API int b200_ppo1_grad(const b200_ppo2_batch *batch, const b200_mlp *actor, const b200_mlp *critic, float std,
                            const float *std_vec, const float *a_min, const float *a_max, float eps_clip,
                            float entropy_coef, float value_coef, float *value, float *grad_actor, float *grad_critic,
                            float *loss_out, void *workspace, size_t workspace_bytes, void *cuda_stream);

/* torch.nn.utils.clip_grad_norm_(params, max_norm) followed by torch.optim.Adam.step() (PPO2.py:118-121,126-129; Adam
 * eps 1e-5, :50-55) as ONE kernel over flat buffers: for each of the n_seg segments (one per net) the global gradient
 * norm is computed in a fixed order, grad is scaled by min(1, max_norm / (norm + 1e-6)) (max_norm <= 0: no clipping)
 * and param, exp_avg (m), exp_avg_sq (v) are updated in place with bias corrections for step number `step` (1-based).
 * grad is first multiplied by grad_scale (1 / world size after a SUM all-reduce of the flat gradient buffer: the DPPO2
 * gradient push, Distributed_PPO2.py:86-104).  Segment j covers elements seg_off[j] .. seg_off[j] + seg_len[j] - 1 of
 * all four buffers and uses learning rate lr[j] (host arrays).  grad_norm_out: device float32 [n_seg] or NULL. */
B200_API int b200_adam_step(int n_seg, const int64_t *seg_off, const int64_t *seg_len, const float *lr, float *param,
                            const float *grad, float *exp_avg, float *exp_avg_sq, int64_t step, float beta1,
                            float beta2, float eps, float max_norm, float grad_scale, float *grad_norm_out,
                            void *cuda_stream);

/* The keyed permutation of [0, B) the kernels above draw mini-batches from, evaluated on the HOST (no GPU involved):
 * out_host[j] = position first + j of the permutation with key perm_key.  For tests and for callers that want to know
 * which samples a mini-batch held. */
B200_API int b200_ppo2_permutation(uint64_t perm_key, int64_t B, int64_t first, int64_t count, int64_t *out_host);

/* The whole K_epochs x mini-batch loop of learn() on one stream without returning to the host between mini-batches
 * (single-GPU training; with several ranks the caller alternates b200_ppo2_grad, the all-reduce and b200_adam_step
 * itself).  Epoch e uses permutation key perm_key + e; mini-batch j covers positions j * mini_batch .. of it (the last
 * one partial, drop_last=False).  `param` is the flat buffer [actor params | critic params] the two b200_mlp structs
 * point into; grad / exp_avg / exp_avg_sq: flat buffers of the same length; `step` is the 1-based Adam step number of
 * the first mini-batch.  loss_out [2]: losses of the last mini-batch. */
B200_API int b200_ppo2_learn(const b200_ppo2_batch *batch, const b200_mlp *actor, const b200_mlp *critic, float std,
                             const float *std_vec, const float *a_min, const float *a_max, float eps_clip,
                             float entropy_coef, int k_epochs, int64_t mini_batch, float lr_actor, float lr_critic,
                             float beta1, float beta2, float adam_eps, float max_norm, int64_t step, float *param,
                             float *grad, float *exp_avg, float *exp_avg_sq, float *loss_out, void *workspace,
                             size_t workspace_bytes, void *cuda_stream);

/* ------------------------------------------------------------- DQN / Double DQN (K-DQN) */

/* Epsilon-greedy action of n instances from a Q-net (tanh hidden layers, identity head: q->out_act must be 0;
 * A = q->dims[q->n_layers] <= 64 actions): obs [S][n] float32 field-major (a row of the replay ring or an env's policy
 * observation).  greedy = argmax_a Q(obs)[a] (lowest index on ties, a NaN output wins as in torch.argmax); with
 * probability epsilon the instance takes a uniform index in [0, A) instead, drawn from ONE Philox4x32-10 block keyed by
 * (seed, offset + i, step) in the key domain 0x44514E41 (csrc/learn.cu states the counter layout and the mapping bit for
 * bit).  Writes action_index [n] int32, action_value [n] = table[action_index] (table: device float32 [A], the float32
 * image of the env's action_space, so that action_value is the env's action buffer [1][n]) and, if q_out is given,
 * q_out [A][n].  Errors, all returned before any CUDA call: B200ENV_ENULL (q, obs, table, action_index, action_value or a
 * weight / bias pointer NULL), B200ENV_ESIZE (n <= 0 or >= 2^31; > 4 layers, a layer or state_dim > 64, > 64 actions),
 * B200ENV_EPARAMS (epsilon outside [0, 1] or NaN, q->out_act != 0, an output overlapping an input or another output). */
B200_API int b200_dqn_act(int64_t n, const b200_mlp *q, const float *obs, const float *table, float epsilon,
                          uint64_t seed, uint64_t step, int64_t offset, int32_t *action_index, float *action_value,
                          float *q_out, void *cuda_stream);

/* The replay ring: R rows of s [R][S][N], r [R][N], s_ [R][S][N] float32, a [R][N] int32 and done [R][N] uint8 (the
 * rollout's is_terminal: terminal states AND time-outs end the bootstrap).  A mini-batch is `count` samples drawn
 * uniformly WITH replacement over the valid_rows newest rows: sample b in [0, valid_rows N) is row
 * (newest_row - b / N) mod R, instance b % N, b from a keyed 64-bit hash of (sample_key, j) and a multiply-high; `index`
 * (device int64 [count] of ring positions row * N + i) overrides the draw.  1 <= valid_rows <= R - 1. */
typedef struct b200_dqn_batch {
    int64_t R, N;
    const float *s, *r, *s_;
    const int32_t *a;
    const uint8_t *done;
    int64_t newest_row, valid_rows, count;
    const int64_t *index;
    uint64_t sample_key;
} b200_dqn_batch;

/* Device bytes of the workspace of b200_dqn_grad for this net and mini-batch size (0 for a net it cannot hold). */
B200_API size_t b200_dqn_workspace_bytes(const b200_mlp *q, int64_t count);

/* One DQN / Double DQN gradient:  y = r + gamma (1 - done) Q_next  (done: y = r exactly), with
 *   DQN         Q_next = max_a Q_target(s', a)
 *   Double DQN  Q_next = Q_target(s', argmax_a Q(s', a))          (double_q != 0)
 * loss = mean_j (Q(s_j)[a_j] - y_j)^2;  grad (device float32 [P], torch parameter order of q) = d loss / d theta;
 * loss_out (device float32 [1]).  Three launches: target, gradient (per-block partials, no atomics), the fixed-order
 * reduction: the bits do not depend on scheduling.  The caller then runs b200_adam_step with n_seg = 1.  q and q_target
 * have the same shapes.  Errors, all returned before any CUDA call: B200ENV_ENULL (a pointer NULL; index may be),
 * B200ENV_ESIZE (R < 2, N <= 0, R or N >= 2^31, count <= 0, net limits as b200_dqn_act, workspace too small),
 * B200ENV_EPARAMS (gamma NaN, valid_rows < 1 or > R - 1, newest_row outside [0, R), shapes differ, out_act != 0, grad /
 * loss_out / workspace overlapping an input, a weight or each other). */
B200_API int b200_dqn_grad(const b200_dqn_batch *batch, const b200_mlp *q, const b200_mlp *q_target, float gamma,
                           int double_q, float *grad, float *loss_out, void *workspace, size_t workspace_bytes,
                           void *cuda_stream);

/* The mini-batch sampler of b200_dqn_grad on the HOST: out_host[j] = ring position (row * N + i) of sample first + j. */
B200_API int b200_dqn_sample_indices(uint64_t sample_key, int64_t newest_row, int64_t valid_rows, int64_t R, int64_t N,
                                     int64_t first, int64_t count, int64_t *out_host);

/* ------------------------------------------------------------- diagnostics */

/* Measures the FP64 (dtype = B200ENV_F64) or FP32 vector FMA peak of the current device in TFLOP/s (2 flops per
 * FMA) with an 8-way independent FMA chain per thread: the roofline denominator of the compute-bound env kernels,
 * which MEASURED_PEAKS.json does not carry.  Blocks until done.  Not on the hot path. */
B200_API int b200_measure_fma_peak(int dtype, int iters, double *tflops, void *cuda_stream);

/* Element-wise evaluation of the in-house fp64 math used by the kernels (csrc/fastmath64.cuh), for accuracy tests:
 * func 0 sincos (out0 = sin, out1 = cos), 1 exp, 2 log, 3 tanh, 4 x^a with a read from out1.  Device pointers. */
B200_API int b200_fastmath_eval(int func, int64_t n, const double *x, double *out0, double *out1, void *cuda_stream);

/* One 128 x N x K product (A [128][K], W [N][K] row-major float32 device arrays, D [128][N] out) through the shared-memory
 * descriptors, instruction descriptor, tcgen05.mma / tcgen05.ld sequence of csrc/policy_umma.cu; three_pass = 1: 3xTF32
 * split, 0: one TF32 pass.  N multiple of 16 <= 256, K multiple of 8 <= 64.  For tests/test_umma_gpu.py. */
B200_API int b200_umma_probe(const float *A, const float *W, float *D, int N, int K, int three_pass, void *cuda_stream);

#ifdef __cplusplus
}
#endif
#endif /* B200ENV_H */
