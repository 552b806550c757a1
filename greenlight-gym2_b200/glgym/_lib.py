"""ctypes binding of libglgym.so (C-ABI declared in include/glgym.h).

The library is built in-tree by `make -C greenlight-gym2_b200/csrc` (or `__graft_entry__.build()`); loading fails
loudly if it is missing -- there is no Python / CPU fallback for the env-step path.
"""
import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libglgym.so")
CSRC_DIR = os.path.join(os.path.dirname(_HERE), "csrc")

NX, NU, ND, NP, NINFO, NSTATS, NNOISE = 28, 6, 10, 208, 11, 16, 34

GLG_OK, GLG_ERR_ARG, GLG_ERR_CUDA, GLG_ERR_STATE, GLG_ERR_ALLOC = 0, -1, -2, -3, -4


class GlgConfig(C.Structure):
    """struct glg_config (include/glgym.h)."""
    _fields_ = [
        ("num_envs", C.c_int32), ("device", C.c_int32), ("dt", C.c_double), ("n_sub", C.c_int32), ("N", C.c_int32),
        ("Np", C.c_int32), ("precision", C.c_int32), ("auto_reset", C.c_int32),
        ("u_min", C.c_double * NU), ("u_max", C.c_double * NU), ("delta_u_max", C.c_double),
        ("con_low", C.c_double * 3), ("con_high", C.c_double * 3),
        ("elec_price", C.c_double), ("heating_price", C.c_double), ("co2_price", C.c_double),
        ("fruit_price", C.c_double), ("dmfm", C.c_double), ("fixed_costs", C.c_double),
        ("uncertainty_scale", C.c_double), ("seed", C.c_uint64), ("env_id_offset", C.c_int64),
        ("role_warps", C.c_int32), ("role_lanes", C.c_int32), ("integrator", C.c_int32), ("reserved2", C.c_int32),
        ("obs_modules", C.c_int32 * 8),
    ]


class GlgRolloutConfig(C.Structure):
    """struct glg_rollout_config (include/glgym.h)."""
    _fields_ = [("n_steps", C.c_int32), ("training", C.c_int32), ("norm_obs", C.c_int32), ("norm_reward", C.c_int32),
                ("gamma", C.c_double), ("gae_lambda", C.c_double), ("clip_obs", C.c_double), ("clip_reward", C.c_double),
                ("epsilon", C.c_double)]


class GlgReplayConfig(C.Structure):
    """struct glg_replay_config (include/glgym.h)."""
    _fields_ = [("buffer_size", C.c_int64), ("training", C.c_int32), ("norm_obs", C.c_int32), ("norm_reward", C.c_int32),
                ("reserved", C.c_int32), ("gamma", C.c_double), ("clip_obs", C.c_double), ("clip_reward", C.c_double),
                ("epsilon", C.c_double), ("seed", C.c_uint64)]


class GlgPlanConfig(C.Structure):
    """struct glg_plan_config (include/glgym.h)."""
    _fields_ = [("horizon", C.c_int32), ("n_candidates", C.c_int32), ("n_elites", C.c_int32), ("n_iterations", C.c_int32),
                ("gamma", C.c_double), ("init_std", C.c_double), ("seed", C.c_uint64)]


class GlgEstConfig(C.Structure):
    """struct glg_est_config (include/glgym.h)."""
    _fields_ = [("alpha", C.c_double), ("beta", C.c_double), ("kappa", C.c_double), ("meas_mask", C.c_int32), ("reserved", C.c_int32),
                ("p0_std", C.c_double * NX), ("q_std", C.c_double * NX), ("r_std", C.c_double * 7)]


class GlgEnvState(C.Structure):
    """struct glg_env_state (include/glgym.h): host pointers, NULL = skip."""
    _fields_ = [("x", C.c_void_p), ("u", C.c_void_p), ("timestep", C.c_void_p), ("table", C.c_void_p), ("time", C.c_void_p),
                ("step_ctr", C.c_void_p), ("ep_return", C.c_void_p), ("ep_len", C.c_void_p), ("ep_info", C.c_void_p)]


# name -> (restype, argtypes); every symbol include/glgym.h declares
_VP, _DP, _FP, _IP, _U8P = C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p
SIGNATURES = {
    "glg_default_config": (None, [C.POINTER(GlgConfig)]),
    "glg_create": (C.c_int, [C.POINTER(GlgConfig), C.POINTER(C.c_void_p)]),
    "glg_destroy": (None, [C.c_void_p]),
    "glg_last_error": (C.c_char_p, [C.c_void_p]),
    "glg_set_params": (C.c_int, [C.c_void_p, _DP]),
    "glg_set_weather": (C.c_int, [C.c_void_p, _DP, C.c_int32, C.c_int32, _DP]),
    "glg_set_reset_tables": (C.c_int, [C.c_void_p, _IP, C.c_int32]),
    "glg_reset": (C.c_int, [C.c_void_p, _U8P, _IP, _VP]),
    "glg_step": (C.c_int, [C.c_void_p, _FP, _DP, _VP]),
    "glg_step_raw_control": (C.c_int, [C.c_void_p, _DP, _DP, _VP]),
    "glg_set_rule_controller": (C.c_int, [C.c_void_p, _DP]),
    "glg_step_rule_based": (C.c_int, [C.c_void_p, _DP, _VP]),
    "glg_rule_control_batch": (C.c_int, [_DP, _DP, _DP, _DP, _DP, _DP, C.c_int32, C.c_int32, _VP]),
    "glg_rule_controls": (C.c_int, [C.c_void_p, _DP, _DP, _VP]),
    "glg_step_host": (C.c_int, [C.c_void_p, _FP, _FP, _DP, _U8P]),
    "glg_step_host_split": (C.c_int, [C.c_void_p, _FP, _FP, _IP, _IP, _DP, _U8P]),
    "glg_set_host_obs_mode": (C.c_int, [C.c_void_p, C.c_int32]),
    "glg_host_path_after": (C.c_int, [C.c_void_p, _VP]),
    "glg_obs_dim": (C.c_int32, [C.c_void_p]),
    "glg_obs_dev": (C.c_void_p, [C.c_void_p]),
    "glg_terminal_obs_dev": (C.c_void_p, [C.c_void_p]),
    "glg_reward_dev": (C.c_void_p, [C.c_void_p]),
    "glg_done_dev": (C.c_void_p, [C.c_void_p]),
    "glg_info_dev": (C.c_void_p, [C.c_void_p]),
    "glg_state_dev": (C.c_void_p, [C.c_void_p]),
    "glg_controls_dev": (C.c_void_p, [C.c_void_p]),
    "glg_timestep_dev": (C.c_void_p, [C.c_void_p]),
    "glg_table_dev": (C.c_void_p, [C.c_void_p]),
    "glg_time_dev": (C.c_void_p, [C.c_void_p]),
    "glg_stats_dev": (C.c_void_p, [C.c_void_p]),
    "glg_clear_stats": (C.c_int, [C.c_void_p, _VP]),
    "glg_set_state": (C.c_int, [C.c_void_p, _DP, _DP, _IP]),
    "glg_get_state": (C.c_int, [C.c_void_p, _DP, _DP, _IP]),
    "glg_set_seed": (C.c_int, [C.c_void_p, C.c_uint64]),
    "glg_get_state_ex": (C.c_int, [C.c_void_p, C.POINTER(GlgEnvState)]),
    "glg_set_state_ex": (C.c_int, [C.c_void_p, C.POINTER(GlgEnvState)]),
    "glg_rollout_create": (C.c_int, [C.c_void_p, C.POINTER(GlgRolloutConfig), C.POINTER(C.c_void_p)]),
    "glg_rollout_destroy": (None, [C.c_void_p]),
    "glg_rollout_store": (C.c_int, [C.c_void_p, C.c_int32, _VP]),
    "glg_rollout_carry": (C.c_int, [C.c_void_p, _VP]),
    "glg_rollout_gae": (C.c_int, [C.c_void_p, _FP, _VP]),
    "glg_rollout_obs_dev": (C.c_void_p, [C.c_void_p]),
    "glg_rollout_rewards_dev": (C.c_void_p, [C.c_void_p]),
    "glg_rollout_starts_dev": (C.c_void_p, [C.c_void_p]),
    "glg_rollout_advantages_dev": (C.c_void_p, [C.c_void_p]),
    "glg_rollout_returns_dev": (C.c_void_p, [C.c_void_p]),
    "glg_rollout_stats_dev": (C.c_void_p, [C.c_void_p]),
    "glg_replay_create": (C.c_int, [C.c_void_p, C.POINTER(GlgReplayConfig), C.POINTER(C.c_void_p)]),
    "glg_replay_destroy": (None, [C.c_void_p]),
    "glg_replay_reset": (C.c_int, [C.c_void_p, _VP]),
    "glg_replay_store": (C.c_int, [C.c_void_p, _FP, _VP]),
    "glg_replay_sample": (C.c_int, [C.c_void_p, C.c_int32, _FP, _FP, _FP, _FP, _FP, _IP, _VP]),
    "glg_replay_size": (C.c_int64, [C.c_void_p]),
    "glg_replay_bytes": (C.c_int64, [C.c_void_p]),
    "glg_replay_obs_dev": (C.c_void_p, [C.c_void_p]),
    "glg_replay_stats_dev": (C.c_void_p, [C.c_void_p]),
    "glg_plan_create": (C.c_int, [C.c_void_p, C.POINTER(GlgPlanConfig), C.POINTER(C.c_void_p)]),
    "glg_plan_destroy": (None, [C.c_void_p]),
    "glg_plan_run": (C.c_int, [C.c_void_p, _FP, _VP]),
    "glg_plan_evaluate": (C.c_int, [C.c_void_p, _FP, _DP, _VP]),
    "glg_plan_shift": (C.c_int, [C.c_void_p, _VP]),
    "glg_plan_run_from": (C.c_int, [C.c_void_p, _DP, _FP, _VP]),
    "glg_plan_mean_dev": (C.c_void_p, [C.c_void_p]),
    "glg_plan_std_dev": (C.c_void_p, [C.c_void_p]),
    "glg_plan_candidates_dev": (C.c_void_p, [C.c_void_p]),
    "glg_plan_returns_dev": (C.c_void_p, [C.c_void_p]),
    "glg_est_create": (C.c_int, [C.c_void_p, C.POINTER(GlgEstConfig), C.POINTER(C.c_void_p)]),
    "glg_est_destroy": (None, [C.c_void_p]),
    "glg_est_reset": (C.c_int, [C.c_void_p, _DP, _VP]),
    "glg_est_update": (C.c_int, [C.c_void_p, _DP, _VP]),
    "glg_est_mean_dev": (C.c_void_p, [C.c_void_p]),
    "glg_est_cov_dev": (C.c_void_p, [C.c_void_p]),
    "glg_est_innovation_dev": (C.c_void_p, [C.c_void_p]),
    "glg_est_sigma_dev": (C.c_void_p, [C.c_void_p]),
    "glg_est_status_dev": (C.c_void_p, [C.c_void_p]),
    "glg_smooth_create": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_void_p)]),
    "glg_smooth_destroy": (None, [C.c_void_p]),
    "glg_smooth_run": (C.c_int, [C.c_void_p, _VP]),
    "glg_smooth_length": (C.c_int32, [C.c_void_p]),
    "glg_smooth_first": (C.c_int32, [C.c_void_p]),
    "glg_smooth_bytes": (C.c_int64, [C.c_void_p]),
    "glg_smooth_mean_dev": (C.c_void_p, [C.c_void_p]),
    "glg_smooth_cov_dev": (C.c_void_p, [C.c_void_p]),
    "glg_smooth_gain_dev": (C.c_void_p, [C.c_void_p]),
    "glg_smooth_filtered_mean_dev": (C.c_void_p, [C.c_void_p]),
    "glg_smooth_filtered_cov_dev": (C.c_void_p, [C.c_void_p]),
    "glg_smooth_prior_mean_dev": (C.c_void_p, [C.c_void_p]),
    "glg_smooth_prior_cov_dev": (C.c_void_p, [C.c_void_p]),
    "glg_smooth_cross_dev": (C.c_void_p, [C.c_void_p]),
    "glg_smooth_status_dev": (C.c_void_p, [C.c_void_p]),
    "glg_smooth_timestep_dev": (C.c_void_p, [C.c_void_p]),
    "glg_est_set_noise": (C.c_int, [C.c_void_p, _DP, _DP, _DP]),
    "glg_em_create": (C.c_int, [C.c_void_p, C.c_int64, C.POINTER(C.c_void_p)]),
    "glg_em_destroy": (None, [C.c_void_p]),
    "glg_em_estep": (C.c_int, [C.c_void_p, _VP]),
    "glg_em_bytes": (C.c_int64, [C.c_void_p]),
    "glg_em_logged": (C.c_int64, [C.c_void_p]),
    "glg_em_chunk_pairs": (C.c_int32, [C.c_void_p]),
    "glg_em_controls_dev": (C.c_void_p, [C.c_void_p]),
    "glg_em_table_dev": (C.c_void_p, [C.c_void_p]),
    "glg_em_measurements_dev": (C.c_void_p, [C.c_void_p]),
    "glg_em_flags_dev": (C.c_void_p, [C.c_void_p]),
    "glg_em_loglik_dev": (C.c_void_p, [C.c_void_p]),
    "glg_em_expectation_dev": (C.c_void_p, [C.c_void_p]),
    "glg_em_prediction_dev": (C.c_void_p, [C.c_void_p]),
    "glg_em_used_dev": (C.c_void_p, [C.c_void_p]),
    "glg_em_env_stats_dev": (C.c_void_p, [C.c_void_p]),
    "glg_em_totals_dev": (C.c_void_p, [C.c_void_p]),
    "glg_nccl_unique_id": (C.c_int, [C.c_void_p]),
    "glg_nccl_init": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]),
    "glg_allreduce_stats": (C.c_int, [C.c_void_p, _VP]),
    "glg_evalf_batch": (C.c_int, [_DP, _DP, _DP, _DP, C.c_int32, _DP, _U8P, C.c_int32, C.c_double, C.c_int32,
                                  C.c_int32, _VP]),
    "glg_evalf_batch_ex": (C.c_int, [_DP, _DP, _DP, _DP, C.c_int32, _DP, _U8P, C.c_int32, C.c_double, C.c_int32,
                                     C.c_int32, C.c_int32, _VP]),
    "glg_rhs_jacobian_batch": (C.c_int, [_DP, _DP, _DP, _DP, C.c_int32, _DP, _DP, _DP, C.c_int32, C.c_int32, _VP]),
    "glg_evalf_jacobian_batch": (C.c_int, [_DP, _DP, _DP, _DP, C.c_int32, _DP, _DP, _DP, _U8P, C.c_int32, C.c_double,
                                           C.c_int32, C.c_int32, C.c_int32, _VP]),
    "glg_linearize": (C.c_int, [C.c_void_p, _DP, _DP, _DP, _DP, _VP]),
    "glg_launch_count": (C.c_int64, [C.c_void_p]),
    "glg_measure_fp64_peak": (C.c_int, [C.c_int32, C.POINTER(C.c_double)]),
    "glg_measure_fp32_peak": (C.c_int, [C.c_int32, C.POINTER(C.c_double)]),
    "glg_debug_math": (C.c_int, [C.c_int32, _DP, _DP, C.c_int32, _VP]),
}

_lib = None


class GlgError(RuntimeError):
    pass


def build(verbose=False):
    """Compile libglgym.so for sm_100a with nvcc (cross-compiles without a GPU)."""
    out = subprocess.run(["make", "-C", CSRC_DIR], capture_output=True, text=True)
    if verbose or out.returncode != 0:
        print(out.stdout[-4000:])
        print(out.stderr[-4000:])
    if out.returncode != 0:
        raise GlgError("building libglgym.so failed")
    return LIB_PATH


def load():
    """Returns the loaded library with all prototypes set; raises if the CUDA extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise GlgError(f"{LIB_PATH} is missing: build it with `make -C {CSRC_DIR}` "
                       "(there is no CPU fallback for the GreenLight env-step path)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, handle=None, what=""):
    if rc != GLG_OK:
        msg = load().glg_last_error(handle)
        raise GlgError(f"{what} failed with status {rc}: {msg.decode() if msg else ''}")
