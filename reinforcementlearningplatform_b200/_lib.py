"""ctypes binding of libb200env.so (C ABI declared in include/b200env.h).

The library is the product: there is no Python/torch fallback.  If the shared
object is missing this module raises, and every env class fails with it.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# B200ENV_LIB selects an alternative build of the same library (A/B experiments with compile-time options)
LIB_PATH = os.environ.get("B200ENV_LIB") or os.path.join(_HERE, "libb200env.so")

# enum b200env_id
CARTPOLE, FAS, SOI, BALLBALANCER, TWOLINK, UGV, UGVO, UAV_ATT, UAV_POS, UAVROBUST, FAS_DISCRETE = range(11)
F64, F32 = 0, 1
AUTO_RESET = 1

ERRORS = {
    0: "ok",
    -1: "B200ENV_EENV: unknown env id / variant",
    -2: "B200ENV_EDTYPE: bad dtype",
    -3: "B200ENV_EPARAMS: params struct size mismatch (ABI drift between Python mirror and library)",
    -4: "B200ENV_ENULL: required pointer is NULL",
    -5: "B200ENV_ECUDA: CUDA launch failed",
    -6: "B200ENV_ESIZE: bad n_envs, or a net the selected K-POLICY kernel cannot hold",
}


class B200EnvError(RuntimeError):
    pass


class IO(C.Structure):
    """struct b200env_io"""
    _fields_ = [(k, C.c_void_p) for k in (
        "state", "time", "episode", "action", "dis", "obs", "next_obs", "reward", "done", "flag", "reset_obs", "work")] + [
        ("io_dtype", C.c_int32), ("pad_", C.c_int32)]


class RolloutSpec(C.Structure):
    """struct b200env_rollout_spec"""
    _fields_ = [(k, C.c_int64) for k in (
        "steps", "action_stride", "dis_stride", "obs_stride", "next_obs_stride", "reward_stride", "done_stride",
        "flag_stride")]


class MLP(C.Structure):
    """struct b200_mlp"""
    _fields_ = [("n_layers", C.c_int32), ("dims", C.c_int32 * 5), ("out_act", C.c_int32), ("pad_", C.c_int32),
                ("w", C.c_void_p * 4), ("b", C.c_void_p * 4)]


class PPO2Batch(C.Structure):
    """struct b200_ppo2_batch"""
    _fields_ = [("T", C.c_int64), ("N", C.c_int64)] + [(k, C.c_void_p) for k in ("s", "a", "a_lp", "adv", "v_target", "index")] + [
        ("first", C.c_int64), ("count", C.c_int64), ("perm_key", C.c_uint64)]


class DQNBatch(C.Structure):
    """struct b200_dqn_batch"""
    _fields_ = [("R", C.c_int64), ("N", C.c_int64)] + [(k, C.c_void_p) for k in ("s", "r", "s_", "a", "done")] + [
        ("newest_row", C.c_int64), ("valid_rows", C.c_int64), ("count", C.c_int64), ("index", C.c_void_p),
        ("sample_key", C.c_uint64)]


class CartPoleParams(C.Structure):
    """struct b200_cartpole_params"""
    _fields_ = [(k, C.c_double) for k in (
        "M", "m", "g", "ell", "kf", "dt", "time_max", "theta_max", "dtheta_max", "x_max", "dx_max",
        "static_gain", "norm_boundless", "theta_term_hi", "theta_term_lo",
        "reset_theta_lo", "reset_theta_hi", "reset_x_lo", "reset_x_hi")] + [
        ("variant", C.c_int32), ("pad_", C.c_int32)]


def _d(name, n=1):
    return (name, C.c_double if n == 1 else C.c_double * n)


class UavParams(C.Structure):
    """struct b200_uav_params"""
    _fields_ = [
        _d("m"), _d("g"), _d("J", 3), _d("kr"), _d("kt"), _d("dt"), _d("time_max"),
        _d("pos_lo", 3), _d("pos_hi", 3), _d("att_lo", 3), _d("att_hi", 3),
        _d("att_zone_min", 3), _d("att_zone_max", 3), _d("t_term"), _d("init_state", 12),
        _d("att_k1", 3), _d("att_k2", 3), _d("att_alpha", 3), _d("att_beta", 3), _d("att_gamma", 3), _d("att_lmd", 3),
        _d("pos_k1", 3), _d("pos_k2", 3), _d("pos_alpha", 3), _d("pos_beta", 3), _d("pos_gamma", 3), _d("pos_lmd", 3),
        _d("Q_e", 3), _d("Q_de", 3), _d("R", 3),
        _d("ref_amplitude", 4), _d("ref_period", 4), _d("ref_bias_a", 4), _d("ref_bias_phase", 4),
        _d("dot_att_ref_limit"), _d("att_limit"), _d("traj_A_hi", 4), _d("traj_T_lo"), _d("traj_T_hi"),
        _d("traj_phase_hi"), _d("init_pos_r", 3), ("random_trajectory", C.c_int32), ("yaw_fixed", C.c_int32),
        ("random_pos0", C.c_int32), ("pad_", C.c_int32)]


def _struct(name, doc, doubles, ints=()):
    fields = [(k, C.c_double) for k in doubles] + [(k, C.c_int32) for k in ints]
    return type(name, (C.Structure,), {"_fields_": fields, "__doc__": doc})


FasParams = _struct("FasParams", "struct b200_fas_params", (
    "L", "k", "mgd", "denom", "dt", "time_max", "min_theta", "max_theta", "min_omega", "max_omega", "static_gain",
    "theta_term_hi", "theta_term_lo", "Q", "R", "reset_lo", "reset_hi"))
FasDiscreteParams = _struct("FasDiscreteParams", "struct b200_fas_discrete_params", (
    "a2", "a1", "L", "denom", "dt", "time_max", "theta_max", "dtheta_max", "static_gain", "theta_out", "Q", "R", "bounce"))
SoiParams = _struct("SoiParams", "struct b200_soi_params", (
    "map_x", "map_y", "target_x", "target_y", "mass", "k", "vmax", "dt", "time_max", "admissible_error", "obs_gain",
    "Q_pos", "Q_vel", "Q_acc", "reset_margin"), ("success_terminal", "pad_"))
BallBalancerParams = _struct("BallBalancerParams", "struct b200_ballbalancer_params", (
    "K", "L", "omega_min", "omega_max", "theta_min", "theta_max", "v_min", "v_max", "dt", "time_max", "static_gain",
    "target", "deg1", "reset_theta_lo", "reset_theta_hi", "reset_pos_lo", "reset_pos_hi", "init_vel"))
TwoLinkParams = _struct("TwoLinkParams", "struct b200_twolink_params", (
    "l", "m", "g", "J", "dt", "time_max", "base_x", "base_y", "theta_max", "miss", "omega_ok", "init_end_x",
    "init_end_y", "r2_lo", "r2_hi", "Q_pos", "Q_omega", "Q_acc"))
UgvParams = _struct("UgvParams", "struct b200_ugv_params", (
    "map_x", "map_y", "target_x", "target_y", "dt", "time_max", "kf", "kt", "e_max", "v_max", "e_phi_max", "omega_max",
    "static_gain", "Q_pos", "Q_vel", "Q_phi", "Q_omega", "reset_d0"), ("bidirectional", "pad_"))

UgvoParams = _struct("UgvoParams", "struct b200_ugvo_params", (
    "map_x", "map_y", "dt", "time_max", "kf", "kt", "e_max", "v_max", "e_phi_max", "omega_max", "static_gain",
    "r_vehicle", "laser_dis", "laser_blind", "laser_range", "Q_pos", "Q_vel", "Q_phi", "Q_omega", "safety_dis_obs",
    "safety_dis_st", "r_min", "r_max", "st_margin"), ("n_rays", "obs_num", "variant", "pad_"))

class UavRobustParams(C.Structure):
    """struct b200_uavrobust_params"""
    _fields_ = [
        _d("m"), _d("g"), _d("J", 3), _d("kr"), _d("kt"), _d("dt"), _d("time_max"), _d("t_term"),
        _d("pos_zone_min", 3), _d("pos_zone_max", 3), _d("att_zone_min", 3), _d("att_zone_max", 3),
        _d("pos0", 3), _d("vel0", 3), _d("angle0", 3), _d("pqr0", 3),
        _d("att_k1", 3), _d("att_k2", 3), _d("att_alpha", 3), _d("att_beta", 3), _d("att_gamma", 3), _d("att_lmd", 3),
        _d("att_saturation", 3), _d("e_pos_span", 3), _d("vel_span", 3), _d("e_att_span", 3), _d("e_dot_att_span_neg", 3),
        _d("dot_att_min", 3), _d("dot_att_max", 3), _d("static_gain"), _d("Qx"), _d("Qv"), _d("R"),
        _d("ref_bias_a", 3), _d("target_lo", 3), _d("target_hi", 3), _d("sig_A_hi", 3), _d("sig_T_lo"), _d("sig_T_hi"),
        _d("sig_phase_hi"), _d("init_pos_r"), ("variant", C.c_int32), ("pad_", C.c_int32)]


PARAMS_OF = {UAVROBUST: UavRobustParams, FAS_DISCRETE: FasDiscreteParams, UGVO: UgvoParams, CARTPOLE: CartPoleParams, UAV_ATT: UavParams, UAV_POS: UavParams, FAS: FasParams, SOI: SoiParams,
             BALLBALANCER: BallBalancerParams, TWOLINK: TwoLinkParams, UGV: UgvParams}

_lib = None


def load() -> C.CDLL:
    """Load libb200env.so once; raise loudly if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise B200EnvError(
            f"{LIB_PATH} not found: the CUDA engine is not built. Run "
            "`python -c 'import __graft_entry__ as g; g.build()'` (or `make -C "
            "reinforcementlearningplatform_b200/csrc`). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, u32, u64, sz = C.c_void_p, C.c_int, C.c_int64, C.c_uint32, C.c_uint64, C.c_size_t
    ip = C.POINTER(C.c_int)
    lib.b200env_version.restype = C.c_char_p
    lib.b200env_version.argtypes = []
    lib.b200env_last_cuda_error.restype = i32
    lib.b200env_last_cuda_error.argtypes = []
    lib.b200env_params_bytes.restype = sz
    lib.b200env_params_bytes.argtypes = [i32]
    lib.b200env_dims.restype = i32
    lib.b200env_dims.argtypes = [i32, i32, ip, ip, ip, ip]
    lib.b200env_state_layout.restype = i32
    lib.b200env_state_layout.argtypes = [i32, i32, ip, ip]
    lib.b200env_state_elems.restype = sz
    lib.b200env_state_elems.argtypes = [i32, i32, i64]
    lib.b200env_step.restype = i32
    lib.b200env_step.argtypes = [i32, i32, i64, vp, sz, C.POINTER(IO), u32, u64, i64, vp]
    lib.b200env_rollout.restype = i32
    lib.b200env_rollout.argtypes = [i32, i32, i64, vp, sz, C.POINTER(IO), C.POINTER(RolloutSpec), u32, u64, i64, vp]
    lib.b200env_reset.restype = i32
    lib.b200env_reset.argtypes = [i32, i32, i64, vp, sz, C.POINTER(IO), vp, u64, i64, vp]
    lib.b200env_observe.restype = i32
    lib.b200env_observe.argtypes = [i32, i32, i64, vp, sz, C.POINTER(IO), vp]
    f64 = C.c_double
    lib.b200_gae.restype = i32
    lib.b200_gae.argtypes = [i64, i64, vp, vp, vp, vp, vp, f64, f64, i32, vp, vp, vp, vp, sz, vp]
    lib.b200_gae_flags.restype = i32
    lib.b200_gae_flags.argtypes = [i64, i64, vp, vp, vp, vp, vp, i32, f64, f64, i32, vp, vp, vp, vp, sz, vp]
    lib.b200_gae_scratch_bytes.restype = sz
    lib.b200_gae_scratch_bytes.argtypes = [i64]
    lib.b200_adv_normalize.restype = i32
    lib.b200_adv_normalize.argtypes = [i64, vp, vp, f64, vp]
    lib.b200_mc_returns.restype = i32
    lib.b200_mc_returns.argtypes = [i32, i64, i64, vp, vp, f64, vp, vp]
    lib.b200_mc_returns_stats.restype = i32
    lib.b200_mc_returns_stats.argtypes = [i32, i64, i64, vp, vp, f64, vp, vp, vp, sz, vp]
    lib.b200_episode_scratch_bytes.restype = sz
    lib.b200_episode_scratch_bytes.argtypes = [i64]
    lib.b200_episode_scan.restype = i32
    lib.b200_episode_scan.argtypes = [i32, i64, i64, vp, vp, vp, vp, vp, vp, vp, vp, i32, vp, vp, sz, vp]
    lib.b200_norm_scratch_bytes.restype = sz
    lib.b200_norm_scratch_bytes.argtypes = [i32]
    lib.b200_norm_seq.restype = i32
    lib.b200_norm_seq.argtypes = [i32, i64, i32, vp, vp, vp, i32, f64, vp]
    lib.b200_norm_batch_stats.restype = i32
    lib.b200_norm_batch_stats.argtypes = [i32, i64, i32, vp, vp, vp, vp, vp]
    lib.b200_norm_merge_apply.restype = i32
    lib.b200_norm_merge_apply.argtypes = [i32, i64, i32, vp, vp, vp, i32, vp, vp, i32, f64, vp]
    lib.b200_norm_rows_prefix.restype = i32
    lib.b200_norm_rows_prefix.argtypes = [i32, vp, i32, vp, vp, vp, vp]
    lib.b200_policy_forward.restype = i32
    lib.b200_policy_forward.argtypes = [i64, vp, vp, vp, vp, vp, C.c_float, vp, u64, u64, i64, i32, vp, vp, vp, vp, vp]
    lib.b200_policy_workspace_bytes.restype = sz
    lib.b200_policy_workspace_bytes.argtypes = [vp, vp]
    lib.b200_policy_pack.restype = i32
    lib.b200_policy_pack.argtypes = [vp, vp, vp, sz, vp]
    lib.b200_policy_forward_packed.restype = i32
    lib.b200_policy_forward_packed.argtypes = [i64, vp, vp, vp, sz, vp, vp, vp, C.c_float, vp, vp, u64, u64, i64, vp, vp, vp,
                                               vp, vp]
    f32 = C.c_float
    lib.b200_ppo2_workspace_bytes.restype = sz
    lib.b200_ppo2_workspace_bytes.argtypes = [vp, vp]
    lib.b200_ppo2_grad.restype = i32
    lib.b200_ppo2_grad.argtypes = [vp, vp, vp, f32, vp, vp, vp, f32, f32, vp, vp, vp, vp, sz, vp]
    lib.b200_ppo1_grad.restype = i32
    lib.b200_ppo1_grad.argtypes = [vp, vp, vp, f32, vp, vp, vp, f32, f32, f32, vp, vp, vp, vp, vp, sz, vp]
    lib.b200_adam_step.restype = i32
    lib.b200_adam_step.argtypes = [i32, C.POINTER(i64), C.POINTER(i64), C.POINTER(f32), vp, vp, vp, vp, i64, f32, f32, f32,
                                   f32, f32, vp, vp]
    lib.b200_ppo2_permutation.restype = i32
    lib.b200_ppo2_permutation.argtypes = [u64, i64, i64, i64, C.POINTER(i64)]
    lib.b200_ppo2_learn.restype = i32
    lib.b200_ppo2_learn.argtypes = [vp, vp, vp, f32, vp, vp, vp, f32, f32, i32, i64, f32, f32, f32, f32, f32, f32, i64, vp,
                                    vp, vp, vp, vp, vp, sz, vp]
    lib.b200_dqn_act.restype = i32
    lib.b200_dqn_act.argtypes = [i64, vp, vp, vp, f32, u64, u64, i64, vp, vp, vp, vp]
    lib.b200_dqn_workspace_bytes.restype = sz
    lib.b200_dqn_workspace_bytes.argtypes = [vp, i64]
    lib.b200_dqn_grad.restype = i32
    lib.b200_dqn_grad.argtypes = [vp, vp, vp, f32, i32, vp, vp, vp, sz, vp]
    lib.b200_dqn_sample_indices.restype = i32
    lib.b200_dqn_sample_indices.argtypes = [u64, i64, i64, i64, i64, i64, i64, C.POINTER(i64)]
    lib.b200_umma_probe.restype = i32
    lib.b200_umma_probe.argtypes = [vp, vp, vp, i32, i32, i32, vp]
    lib.b200_fastmath_eval.restype = i32
    lib.b200_fastmath_eval.argtypes = [i32, i64, vp, vp, vp, vp]
    lib.b200_measure_fma_peak.restype = i32
    lib.b200_measure_fma_peak.argtypes = [i32, i32, C.POINTER(C.c_double), vp]
    _lib = lib
    return lib


def measure_fma_peak(dtype_code: int = F64, iters: int = 20000) -> float:
    """TFLOP/s of the FP64/FP32 vector FMA pipe of the current CUDA device (diagnostic, include/b200env.h)."""
    out = C.c_double()
    check(load().b200_measure_fma_peak(dtype_code, iters, C.byref(out), None), "b200_measure_fma_peak")
    return out.value


def check(rc: int, what: str) -> None:
    if rc != 0:
        extra = ""
        if rc == -5:
            extra = f" (cudaError {load().b200env_last_cuda_error()})"
        raise B200EnvError(f"{what}: {ERRORS.get(rc, rc)}{extra}")


def state_layout(env_id: int, variant: int = 0):
    """(block, slots) of the persistent state buffer: block == 0 -> field-major [slots = state_fields][n]."""
    b, s = C.c_int(), C.c_int()
    check(load().b200env_state_layout(env_id, variant, C.byref(b), C.byref(s)), "b200env_state_layout")
    return b.value, s.value


def dims(env_id: int, variant: int = 0):
    sf, od, ad, dd = C.c_int(), C.c_int(), C.c_int(), C.c_int()
    check(load().b200env_dims(env_id, variant, C.byref(sf), C.byref(od), C.byref(ad), C.byref(dd)), "b200env_dims")
    return sf.value, od.value, ad.value, dd.value
