"""ctypes binding of ``libmyo_b200.so`` (C ABI declared in ``include/myo_b200.h``).

There is no CPU path behind this module: if the CUDA library has not been built
(``python -c "import __graft_entry__ as g; g.build()"``) importing the product fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmyo_b200.so")

MYO_MAX_OVERRIDE = 4
MYO_INFO_TERMS = 12
MYO_MAX_ROT_RANGES = 4
MYO_MAX_OBS_KEYS = 16
TASK_STATE_I, TASK_STATE_F = 4, 8
TASK_NONE, TASK_POSE, TASK_BAODING, TASK_REORIENT, TASK_REACH = 0, 1, 2, 3, 4
PARAM_BODY_MASS, PARAM_GEOM_SIZE, PARAM_GEOM_FRICTION, PARAM_SITE_POS, PARAM_BODY_POS, PARAM_BODY_MAT = 0, 1, 2, 3, 4, 5
PARAM_NCOMP = {0: 1, 1: 3, 2: 3, 3: 3, 4: 3, 5: 9}

STAGES = {
    "xpos": 0, "xmat": 1, "site_xpos": 2, "ten_length": 3, "ten_J": 4, "qM": 5, "qfrc_bias": 6,
    "qfrc_passive": 7, "qfrc_actuator": 8, "actuator_force": 9, "qacc_smooth": 10, "qacc": 11, "ncon": 12,
    "contact_geoms": 13, "contact_dist": 14, "nefc": 15, "efc_type_id": 16, "efc_J": 17, "efc_aref": 18,
    "efc_D": 19, "efc_force": 20, "qfrc_constraint": 21, "act_dot": 22, "solver_iter": 23, "status": 24,
}
INT_STAGES = {"ncon", "contact_geoms", "nefc", "efc_type_id", "solver_iter", "status"}


class TaskCfg(C.Structure):
    """Mirror of ``struct myo_task_cfg``."""

    _fields_ = [
        ("kind", C.c_int32), ("frame_skip", C.c_int32), ("max_episode_steps", C.c_int32),
        ("normalize_act", C.c_int32), ("auto_reset", C.c_int32), ("solver_iterations", C.c_int32),
        ("solver_tolerance", C.c_float), ("rwd_weight", C.c_float * MYO_INFO_TERMS),
        ("drop_th", C.c_float), ("proximity_th", C.c_float),
        ("goal_time_period", C.c_float * 2), ("goal_xrange", C.c_float * 2), ("goal_yrange", C.c_float * 2),
        ("obj_size_range", C.c_float * 2), ("obj_mass_range", C.c_float * 2), ("obj_friction_change", C.c_float * 3),
        ("task_choice_random", C.c_int32), ("fixed_task", C.c_int32),
        ("overlap_probability", C.c_float), ("limit_init_angle", C.c_float), ("noise_fingers", C.c_float),
        ("center_pos", C.c_float * 2), ("randomize_physics", C.c_int32),
        ("ball_body", C.c_int32 * 2), ("ball_geom", C.c_int32 * 2), ("ball_site", C.c_int32 * 2),
        ("target_site", C.c_int32 * 2), ("ball_qposadr", C.c_int32 * 2), ("ball_dofadr", C.c_int32 * 2),
        ("pose_thd", C.c_float), ("far_th", C.c_float), ("target_distance", C.c_float),
        ("reset_type", C.c_int32), ("target_type", C.c_int32), ("n_target_jnt", C.c_int32),
        ("target_jnt_ids", C.c_int32 * 64), ("target_jnt_range", (C.c_float * 2) * 64),
        ("target_jnt_value", C.c_float * 64),
        ("n_ovr_body", C.c_int32), ("ovr_body", C.c_int32 * MYO_MAX_OVERRIDE),
        ("n_ovr_geom", C.c_int32), ("ovr_geom", C.c_int32 * MYO_MAX_OVERRIDE),
        ("n_ovr_site", C.c_int32), ("ovr_site", C.c_int32 * MYO_MAX_OVERRIDE),
        ("clip_actions", C.c_int32),
        ("enable_rsi", C.c_int32), ("rsi_probability", C.c_float), ("balls_overlap", C.c_int32),
        ("beta_init_angle", C.c_float * 2), ("beta_ball_size", C.c_float * 2), ("beta_ball_mass", C.c_float * 2),
        ("p1_reset", C.c_int32), ("noise_palm", C.c_float), ("noise_balls", C.c_float),
        ("goal_pos", C.c_float * 2), ("goal_rot", C.c_float * 2), ("obj_size_change", C.c_float), ("pos_th", C.c_float), ("rot_th", C.c_float),
        ("n_goal_rot", C.c_int32 * 3), ("goal_rot_axis", ((C.c_float * 2) * MYO_MAX_ROT_RANGES) * 3),
        ("object_body", C.c_int32), ("goal_body", C.c_int32), ("object_site", C.c_int32), ("goal_site", C.c_int32),
        ("object_geom0", C.c_int32), ("object_ngeom", C.c_int32), ("object_qposadr", C.c_int32), ("object_dofadr", C.c_int32),
        ("goal_init_pos", C.c_float * 3), ("goal_obj_offset", C.c_float * 3),
        ("n_ovr_bodypose", C.c_int32), ("ovr_bodypose", C.c_int32 * MYO_MAX_OVERRIDE),
        ("sds_distance", C.c_float), ("weight_body", C.c_int32), ("weight_geom", C.c_int32), ("weight_range", C.c_float * 2),
        ("reach_nsite", C.c_int32), ("reach_tip_site", C.c_int32 * MYO_MAX_OVERRIDE), ("reach_target_site", C.c_int32 * MYO_MAX_OVERRIDE),
        ("reach_range", ((C.c_float * 3) * 2) * MYO_MAX_OVERRIDE), ("reach_near_th", C.c_float), ("reach_far_steps", C.c_int32),
        ("n_obs_keys", C.c_int32), ("obs_keys", C.c_int32 * MYO_MAX_OBS_KEYS), ("reward_sparse", C.c_int32),
    ]


class PPOHyper(C.Structure):
    """Mirror of ``struct myo_ppo_hyper``."""

    _fields_ = [("clip_range", C.c_float), ("clip_range_vf", C.c_float), ("ent_coef", C.c_float), ("vf_coef", C.c_float),
                ("normalize_advantage", C.c_int32)]


class PolicyCfg(C.Structure):
    _fields_ = [
        ("obs_dim", C.c_int32), ("act_dim", C.c_int32), ("lstm_hidden", C.c_int32),
        ("n_pi_layers", C.c_int32), ("pi_layers", C.c_int32 * 4),
        ("n_vf_layers", C.c_int32), ("vf_layers", C.c_int32 * 4),
        ("use_sde", C.c_int32),
    ]


# every symbol include/myo_b200.h declares: name -> (restype, argtypes)
_vp, _i, _ip, _cp, _fp = C.c_void_p, C.c_int, C.POINTER(C.c_int), C.c_char_p, C.c_void_p
SIGNATURES = {
    "myo_last_error": (C.c_char_p, []),
    "myo_version": (C.c_char_p, []),
    "myo_model_load_mjb": (_i, [_cp, C.POINTER(_vp)]),
    "myo_model_load_mjb_mem": (_i, [_vp, C.c_size_t, C.POINTER(_vp)]),
    "myo_model_free": (None, [_vp]),
    "myo_model_size": (_i, [_vp, _cp, _ip]),
    "myo_model_opt": (_i, [_vp, _cp, C.POINTER(C.c_double)]),
    "myo_model_array": (_i, [_vp, _cp, C.POINTER(_vp), _ip, _ip, _ip]),
    "myo_model_name2id": (_i, [_vp, _cp, _cp]),
    "myo_model_id2name": (C.c_char_p, [_vp, _cp, _i]),
    "myo_model_check": (_i, [_vp, C.c_char_p, C.c_size_t]),
    "myo_task_cfg_default": (_i, [_vp, _i, C.POINTER(TaskCfg)]),
    "myo_batch_create": (_i, [_vp, _i, _i, C.POINTER(TaskCfg), C.c_uint64, C.POINTER(_vp)]),
    "myo_batch_destroy": (None, [_vp]),
    "myo_batch_dims": (_i, [_vp, _ip, _ip, _ip, _ip, _ip, _ip, _ip]),
    "myo_batch_launch_info": (_i, [_vp, _ip, _ip, _ip, _ip]),
    "myo_batch_reset": (_i, [_vp, _vp, _fp, _vp]),
    "myo_batch_set_state": (_i, [_vp, _fp, _fp, _fp, _fp, _vp]),
    "myo_batch_get_state": (_i, [_vp, _fp, _fp, _fp, _fp, _vp]),
    "myo_batch_set_param": (_i, [_vp, _i, _i, _fp, _vp]),
    "myo_batch_get_param": (_i, [_vp, _i, _i, _fp, _vp]),
    "myo_batch_get_task_state": (_i, [_vp, _vp, _fp, _fp, _vp]),
    "myo_batch_set_task_state": (_i, [_vp, _vp, _fp, _fp, _vp]),
    "myo_batch_step": (_i, [_vp, _fp, _fp, _fp, _vp, _vp, _fp, _fp, _vp]),
    "myo_batch_mj_step": (_i, [_vp, _fp, _i, _vp]),
    "myo_batch_forward": (_i, [_vp, _fp, _vp]),
    "myo_batch_get_obs": (_i, [_vp, _fp, _vp]),
    "myo_batch_stage_dump": (_i, [_vp, _i, _vp, _ip, _vp]),
    "myo_batch_status": (_i, [_vp, _ip, _vp]),
    "myo_batch_launch_count": (C.c_int64, [_vp]),
    "myo_fp32_fma_peak": (_i, [_i, C.POINTER(C.c_double)]),
    "myo_policy_create": (_i, [C.POINTER(PolicyCfg), _i, _i, C.POINTER(_vp)]),
    "myo_policy_destroy": (None, [_vp]),
    "myo_policy_set_weight": (_i, [_vp, _cp, _fp, C.c_int64, _vp]),
    "myo_policy_forward": (_i, [_vp, _i, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _vp]),
    "myo_policy_set_obs_norm": (_i, [_vp, _fp, _fp, C.c_float, C.c_float, _vp]),
    "myo_policy_seed": (_i, [_vp, C.c_uint64]),
    "myo_policy_set_precision": (_i, [_vp, _i]),
    "myo_policy_launch_count": (C.c_int64, [_vp]),
    "myo_policy_set_latent_out": (_i, [_vp, _fp]),
    "myo_sde_reset_noise": (_i, [_vp, _fp, _fp, _i, _i, _i, C.c_uint64, C.c_uint32, _vp]),
    "myo_sde_sample": (_i, [_fp, _i, _vp, _fp, _fp, _fp, _i, _i, _i, _vp]),
    "myo_running_moments_scratch": (_i, [_i, _i]),
    "myo_running_moments_update": (_i, [_vp, _fp, _i, _i, _vp, _fp, _fp, _vp]),
    "myo_running_moments_export": (_i, [_vp, _i, _fp, _fp, _vp]),
    "myo_vecnorm_reward": (_i, [_vp, _vp, _fp, _vp, _fp, _i, C.c_double, C.c_double, C.c_double, _i, _i, _vp, _vp]),
    "myo_gae": (_i, [_fp, _fp, _vp, _fp, _vp, _i, _i, C.c_float, C.c_float, _fp, _fp, _vp]),
    "myo_normalize_obs": (_i, [_fp, _fp, _fp, C.c_float, C.c_float, _fp, _i, _i, _vp]),
    "myo_ppo_create": (_i, [C.POINTER(PolicyCfg), _i, _i, _i, _i, C.POINTER(_vp)]),
    "myo_ppo_destroy": (None, [_vp]),
    "myo_ppo_param_count": (C.c_int64, [_vp]),
    "myo_ppo_param_offset": (_i, [_vp, _cp, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "myo_ppo_minibatch_grad": (_i, [_vp, _fp, _i, _i, _vp, _i, _fp, _fp, _vp, _fp, _fp, _fp, _fp, _fp, _fp, C.POINTER(PPOHyper), _fp, _fp, _vp]),
    "myo_ppo_adam_step": (_i, [_vp, _fp, _fp, _fp, _fp, _i, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, _fp, _vp]),
    "myo_ppo_launch_count": (C.c_int64, [_vp]),
}


class MyoError(RuntimeError):
    pass


def bind(path: str, only=None) -> C.CDLL:
    """Load a library exporting the C ABI and attach the prototypes (``only``: symbol-name prefix filter)."""
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        if only is not None and not name.startswith(only):
            continue
        fn = getattr(lib, name)   # AttributeError here means the library is missing a declared symbol
        fn.restype = res
        fn.argtypes = args
    return lib


_LIB = None


def lib() -> C.CDLL:
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise MyoError(
                f"{LIB_PATH} is missing: the CUDA extension has not been built "
                "(run `python -c 'import __graft_entry__ as g; g.build()'`). There is no CPU fallback."
            )
        _LIB = bind(LIB_PATH)
    return _LIB


def check(L: C.CDLL, rc: int) -> None:
    if rc != 0:
        raise MyoError(f"myo_b200 error {rc}: {L.myo_last_error().decode(errors='replace')}")
