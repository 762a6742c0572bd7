"""ctypes binding of ``include/rl_mdp_step.h`` (the C-ABI of the CUDA MDP step).

The structures below mirror the header field by field; :func:`load` verifies every ``sizeof`` against
the library (``rl_struct_sizeof``) before anything is called. There is deliberately **no fallback**: if the
shared library is missing or was built for another ABI version this module raises - the product path
never routes through the CPU oracle.
"""

from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import torch

RL_ABI_VERSION = 13
RL_MAX_TASKS = 112
RL_DEBUG_STRIDE = 160
RL_MAX_JOINTS = 64
RL_MAX_BODIES = 64
RL_MAX_TIME_BODIES = 64
RL_MAX_ASSET_BODIES = 64
RL_MAX_REWARD_TERMS = 48
RL_MAX_OBS_TERMS = 12
RL_MAX_DONE_TERMS = 8
RL_MAX_IDX = 32
RL_NUM_OBS_GROUPS = 2
RL_NUM_CMD_UNIFORMS = 7

# enum RlPhase
PHASE_DONES, PHASE_REWARDS, PHASE_COMMAND, PHASE_OBS, PHASE_COMPACT, PHASE_SKIP_DONE_ENVS = 1, 2, 4, 8, 16, 32
PHASE_RESET = 64
PHASE_ALL = 31

# enum RlRewardType (name -> id); checked against the header by tests/test_abi.py
REWARD_TYPES = {
    "is_terminated": 1, "lin_vel_z_l2": 2, "ang_vel_xy_l2": 3, "flat_orientation_l2": 4, "base_height_l2": 5,
    "joint_torques_l2": 6, "joint_vel_l2": 7, "joint_acc_l2": 8, "joint_deviation_l1": 9, "joint_pos_limits": 10,
    "joint_vel_limits": 11, "joint_power": 12, "stand_still": 13, "joint_pos_penalty": 14, "joint_mirror": 15,
    "action_mirror": 16, "action_sync": 17, "action_rate_l2": 18, "undesired_contacts": 19, "contact_forces": 20,
    "track_lin_vel_xy_exp": 21, "track_ang_vel_z_exp": 22, "track_lin_vel_xy_yaw_frame_exp": 23,
    "track_ang_vel_z_world_exp": 24, "feet_air_time": 25, "feet_air_time_positive_biped": 26,
    "feet_air_time_variance": 27, "feet_gait": 28, "feet_contact": 29, "feet_contact_without_cmd": 30,
    "feet_stumble": 31, "feet_slide": 32, "feet_height": 33, "feet_height_body": 34, "feet_distance_y_exp": 35,
    "feet_distance_xy_exp": 36, "upward": 37, "wheel_vel_penalty": 38,
}
OBS_TYPES = {
    "base_lin_vel": 1, "base_ang_vel": 2, "projected_gravity": 3, "generated_commands": 4, "joint_pos_rel": 5,
    "joint_vel_rel": 6, "last_action": 7, "height_scan": 8, "joint_pos_rel_without_wheel": 9, "phase": 10,
}
DONE_TYPES = {"time_out": 1, "terrain_out_of_bounds": 2, "illegal_contact": 3}


class RlRewardTerm(C.Structure):
    _fields_ = [
        ("type", C.c_int32), ("weight", C.c_float), ("p", C.c_float * 6),
        ("joint_mask", C.c_uint64), ("body_mask", C.c_uint64),
        ("n_idx", C.c_int32), ("reserved", C.c_int32),
        ("idx_a", C.c_uint8 * RL_MAX_IDX), ("idx_b", C.c_uint8 * RL_MAX_IDX), ("idx_c", C.c_uint8 * RL_MAX_IDX),
    ]


class RlObsTerm(C.Structure):
    _fields_ = [
        ("type", C.c_int32), ("dim", C.c_int32),
        ("has_noise", C.c_int32), ("noise_lo", C.c_float), ("noise_hi", C.c_float),
        ("has_clip", C.c_int32), ("clip_lo", C.c_float), ("clip_hi", C.c_float),
        ("has_scale", C.c_int32), ("scale", C.c_float),
        ("p", C.c_float * 2), ("zero_mask", C.c_uint64), ("ids", C.c_uint8 * RL_MAX_JOINTS),
    ]


class RlObsGroup(C.Structure):
    _fields_ = [
        ("n_terms", C.c_int32), ("dim", C.c_int32), ("enable_corruption", C.c_int32), ("reserved", C.c_int32),
        ("terms", RlObsTerm * RL_MAX_OBS_TERMS),
    ]


class RlDoneTerm(C.Structure):
    _fields_ = [("type", C.c_int32), ("time_out", C.c_int32), ("p", C.c_float * 4), ("body_mask", C.c_uint64)]


class RlCommandCfg(C.Structure):
    _fields_ = [
        ("resampling_time_lo", C.c_float), ("resampling_time_hi", C.c_float),
        ("rel_standing_envs", C.c_float), ("rel_heading_envs", C.c_float),
        ("heading_command", C.c_int32), ("heading_control_stiffness", C.c_float),
        ("lin_vel_x_lo", C.c_float), ("lin_vel_x_hi", C.c_float),
        ("lin_vel_y_lo", C.c_float), ("lin_vel_y_hi", C.c_float),
        ("ang_vel_z_lo", C.c_float), ("ang_vel_z_hi", C.c_float),
        ("heading_lo", C.c_float), ("heading_hi", C.c_float),
        ("small_cmd_threshold", C.c_float), ("max_command_step", C.c_float),
    ]


class RlActionCfg(C.Structure):
    _fields_ = [
        ("n_actions", C.c_int32), ("has_clip", C.c_int32),
        ("joint_ids", C.c_uint8 * RL_MAX_JOINTS), ("target_kind", C.c_uint8 * RL_MAX_JOINTS),
        ("scale", C.c_float * RL_MAX_JOINTS), ("offset", C.c_float * RL_MAX_JOINTS),
        ("clip_lo", C.c_float * RL_MAX_JOINTS), ("clip_hi", C.c_float * RL_MAX_JOINTS),
    ]


class RlStepSpec(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("num_joints", C.c_int32), ("num_hist_bodies", C.c_int32),
        ("hist_len", C.c_int32), ("num_time_bodies", C.c_int32), ("num_asset_bodies", C.c_int32),
        ("num_rays", C.c_int32), ("num_reward_terms", C.c_int32), ("num_done_terms", C.c_int32),
        ("max_episode_length", C.c_int32), ("step_dt", C.c_float), ("contact_time_abs_tol", C.c_float),
        ("default_joint_pos", C.c_float * RL_MAX_JOINTS), ("default_joint_vel", C.c_float * RL_MAX_JOINTS),
        ("soft_pos_limit_lo", C.c_float * RL_MAX_JOINTS), ("soft_pos_limit_hi", C.c_float * RL_MAX_JOINTS),
        ("soft_vel_limit", C.c_float * RL_MAX_JOINTS),
        ("rewards", RlRewardTerm * RL_MAX_REWARD_TERMS),
        ("dones", RlDoneTerm * RL_MAX_DONE_TERMS),
        ("obs", RlObsGroup * RL_NUM_OBS_GROUPS),
        ("command", RlCommandCfg), ("action", RlActionCfg),
    ]


class RlField(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("env_stride", C.c_int64), ("comp_stride", C.c_int64)]


_STATE_FIELDS = (
    "root_pos_w", "root_quat_w", "root_lin_vel_w", "root_ang_vel_w", "joint_pos", "joint_vel", "joint_acc",
    "applied_torque", "net_forces_w_history", "current_air_time", "last_air_time", "current_contact_time",
    "last_contact_time", "body_pos_w", "body_lin_vel_w", "ray_hits_z", "ray_sensor_pos_z",
)
_MDP_FIELDS = (
    "action", "prev_action", "command", "heading_target", "time_left", "is_heading_env", "is_standing_env",
    "metric_error_vel_xy", "metric_error_vel_yaw", "episode_length", "episode_sums",
)


class RlStateView(C.Structure):
    _fields_ = [(n, RlField) for n in _STATE_FIELDS]


class RlMdpState(C.Structure):
    _fields_ = [(n, RlField) for n in _MDP_FIELDS]


class RlResetLog(C.Structure):
    _fields_ = [("episode_sum_mean", C.c_void_p), ("done_term_count", C.c_void_p), ("metric_mean", C.c_void_p)]


class RlResetStateCfg(C.Structure):
    _fields_ = [
        ("default_root_state", C.c_float * 13), ("pose_lo", C.c_float * 6), ("pose_hi", C.c_float * 6),
        ("vel_lo", C.c_float * 6), ("vel_hi", C.c_float * 6),
        ("joint_pos_scale_lo", C.c_float), ("joint_pos_scale_hi", C.c_float),
        ("joint_vel_scale_lo", C.c_float), ("joint_vel_scale_hi", C.c_float),
    ]


# enum RlActuatorType
ACT_NONE, ACT_IDEAL_PD, ACT_IMPLICIT, ACT_DC_MOTOR = 0, 1, 2, 3
ACTUATOR_TYPES = {"none": ACT_NONE, "ideal_pd": ACT_IDEAL_PD, "implicit": ACT_IMPLICIT, "dc_motor": ACT_DC_MOTOR}


class RlActuatorCfg(C.Structure):
    _fields_ = [
        ("num_joints", C.c_int32), ("reserved", C.c_int32), ("type", C.c_uint8 * RL_MAX_JOINTS),
        ("stiffness", C.c_float * RL_MAX_JOINTS), ("damping", C.c_float * RL_MAX_JOINTS),
        ("effort_limit", C.c_float * RL_MAX_JOINTS), ("saturation_effort", C.c_float * RL_MAX_JOINTS),
        ("velocity_limit", C.c_float * RL_MAX_JOINTS),
    ]


class RlTerrainGrid(C.Structure):
    _fields_ = [("terrain_origins", C.c_void_p), ("num_rows", C.c_int32), ("num_cols", C.c_int32),
                ("col_start", C.c_int32), ("col_end", C.c_int32)]


class RlHeightField(C.Structure):
    _fields_ = [("heights", C.c_void_p), ("num_x", C.c_int32), ("num_y", C.c_int32), ("x0", C.c_float),
                ("y0", C.c_float), ("horizontal_scale", C.c_float), ("num_rays", C.c_int32),
                ("ray_starts", C.c_void_p)]


class RlIntervalEventCfg(C.Structure):
    _fields_ = [("interval_lo", C.c_float), ("interval_hi", C.c_float), ("vel_lo", C.c_float * 6), ("vel_hi", C.c_float * 6)]


# rows of the uniform table of rl_interval_push ([8][N]): timer on reset, timer on fire, velocity x, y, z, roll, pitch, yaw
RL_NUM_INTERVAL_UNIFORMS = 8


class RlStepOut(C.Structure):
    _fields_ = [
        ("obs", C.c_void_p * RL_NUM_OBS_GROUPS), ("obs_pitch", C.c_int64 * RL_NUM_OBS_GROUPS),
        ("reward", C.c_void_p), ("terminated", C.c_void_p), ("truncated", C.c_void_p), ("done_bits", C.c_void_p),
        ("step_reward", RlField), ("reset_ids", C.c_void_p), ("n_reset", C.c_void_p), ("reset_log", RlResetLog),
    ]


class RlRandom(C.Structure):
    _fields_ = [
        ("seed", C.c_uint64), ("step", C.c_uint64), ("step_counter", C.c_void_p), ("env_id_offset", C.c_int64),
        ("cmd_uniforms", C.c_void_p), ("obs_uniforms", C.c_void_p * RL_NUM_OBS_GROUPS),
    ]


_STRUCTS = (RlRewardTerm, RlObsTerm, RlObsGroup, RlDoneTerm, RlCommandCfg, RlActionCfg, RlStepSpec, RlField,
            RlStateView, RlMdpState, RlStepOut, RlRandom, RlResetLog, RlResetStateCfg, RlActuatorCfg, RlTerrainGrid,
            RlHeightField, RlIntervalEventCfg)

EXPORTED_SYMBOLS = (
    "rl_abi_version", "rl_last_error", "rl_struct_sizeof", "rl_tile_record_bytes", "rl_ctx_create", "rl_ctx_destroy",
    "rl_ctx_set_launch_config", "rl_ctx_get_launch_config", "rl_ctx_get_cluster_config", "rl_ctx_set_pdl", "rl_ctx_set_debug_buffer", "rl_ctx_get_schedule",
    "rl_contact_sensor_update", "rl_reset_scene_state", "rl_process_action", "rl_step", "rl_reset_envs", "rl_term_eval",
    "rl_actuator_step", "rl_is_robot_on_terrain", "rl_command_pit_restrict", "rl_height_scan_cast", "rl_derived_views",
    "rl_interval_push",
)

LIB_PATH = Path(__file__).resolve().parent / "_lib" / "libmdpstep.so"
_lib = None


class NativeError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load ``libmdpstep.so`` (built in-tree by ``__graft_entry__.build()`` / ``robot_lab_b200.build``)."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("RL_MDPSTEP_LIB", str(LIB_PATH)))
    if not path.exists():
        raise NativeError(
            f"{path} is missing: build the CUDA extension first (python -m robot_lab_b200.build). "
            "There is no CPU fallback for the MDP step."
        )
    lib = C.CDLL(str(path))
    for sym in EXPORTED_SYMBOLS:
        if not hasattr(lib, sym):
            raise NativeError(f"{path} does not export {sym}")
    lib.rl_abi_version.restype = C.c_int
    lib.rl_last_error.restype = C.c_char_p
    lib.rl_struct_sizeof.restype = C.c_int64
    lib.rl_struct_sizeof.argtypes = [C.c_char_p]
    if lib.rl_abi_version() != RL_ABI_VERSION:
        raise NativeError(f"ABI mismatch: library {lib.rl_abi_version()} vs binding {RL_ABI_VERSION}")
    for st in _STRUCTS:
        want = lib.rl_struct_sizeof(st.__name__.encode())
        if want != C.sizeof(st):
            raise NativeError(f"layout mismatch for {st.__name__}: C {want} vs ctypes {C.sizeof(st)}")
    lib.rl_tile_record_bytes.restype = C.c_int64
    lib.rl_tile_record_bytes.argtypes = [C.POINTER(RlStepSpec)]
    lib.rl_ctx_create.argtypes = [C.POINTER(RlStepSpec), C.c_int, C.POINTER(C.c_void_p)]
    lib.rl_ctx_destroy.argtypes = [C.c_void_p]
    lib.rl_ctx_destroy.restype = None
    lib.rl_ctx_set_launch_config.argtypes = [C.c_void_p, C.c_int, C.c_int]
    lib.rl_ctx_get_launch_config.argtypes = [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.rl_ctx_get_cluster_config.argtypes = [C.c_void_p, C.c_int64, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int64)]
    lib.rl_ctx_set_pdl.argtypes = [C.c_void_p, C.c_int]
    lib.rl_ctx_set_debug_buffer.argtypes = [C.c_void_p, C.c_void_p]
    lib.rl_ctx_get_schedule.argtypes = [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]
    lib.rl_reset_scene_state.argtypes = [C.c_void_p, C.c_int64, C.POINTER(RlResetStateCfg), C.POINTER(RlField),
                                         C.POINTER(RlStateView), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.POINTER(RlRandom), C.c_void_p, C.c_void_p, C.c_void_p]
    lib.rl_actuator_step.argtypes = [C.c_void_p, C.c_int64, C.POINTER(RlActuatorCfg), C.POINTER(RlField),
                                     C.POINTER(RlField), C.POINTER(RlField), C.POINTER(RlStateView),
                                     C.POINTER(RlField), C.c_void_p]
    lib.rl_is_robot_on_terrain.argtypes = [C.c_void_p, C.c_int64, C.POINTER(RlField), C.POINTER(RlTerrainGrid),
                                           C.c_void_p, C.c_void_p]
    lib.rl_command_pit_restrict.argtypes = [C.c_void_p, C.c_int64, C.POINTER(RlField), C.POINTER(RlTerrainGrid),
                                            C.POINTER(RlMdpState), C.c_void_p, C.POINTER(RlRandom), C.c_void_p]
    lib.rl_height_scan_cast.argtypes = [C.c_void_p, C.c_int64, C.POINTER(RlHeightField), C.POINTER(RlStateView),
                                        C.c_void_p]
    lib.rl_derived_views.argtypes = [C.c_void_p, C.c_int64, C.POINTER(RlStateView), C.POINTER(RlField), C.POINTER(RlField),
                                     C.POINTER(RlField), C.POINTER(RlField), C.c_void_p]
    lib.rl_interval_push.argtypes = [C.c_void_p, C.c_int64, C.POINTER(RlIntervalEventCfg), C.c_float, C.c_void_p,
                                     C.POINTER(RlStateView), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.POINTER(RlRandom), C.c_void_p, C.c_void_p]
    lib.rl_contact_sensor_update.argtypes = [C.c_void_p, C.c_int64, C.POINTER(RlField), C.POINTER(RlStateView),
                                             C.POINTER(C.c_int32), C.c_float, C.c_float, C.c_int32, C.c_void_p]
    lib.rl_process_action.argtypes = [C.c_void_p, C.c_int64, C.POINTER(RlField), C.POINTER(RlMdpState),
                                      C.POINTER(RlField), C.POINTER(RlField), C.c_void_p, C.c_void_p]
    lib.rl_step.argtypes = [C.c_void_p, C.c_int64, C.POINTER(RlStateView), C.POINTER(RlMdpState),
                            C.POINTER(RlStepOut), C.POINTER(RlRandom), C.c_uint32, C.c_void_p, C.c_void_p,
                            C.c_void_p]
    lib.rl_reset_envs.argtypes = [C.c_void_p, C.c_int64, C.POINTER(RlMdpState), C.c_void_p, C.POINTER(RlRandom),
                                  C.POINTER(RlResetLog), C.c_void_p, C.c_void_p, C.c_void_p]
    lib.rl_term_eval.argtypes = [C.c_void_p, C.c_int64, C.POINTER(RlRewardTerm), C.POINTER(RlStateView),
                                 C.POINTER(RlMdpState), C.c_void_p, C.c_void_p, C.c_void_p]
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().rl_last_error().decode(errors="replace")
        raise NativeError(f"rl_* call failed ({rc}): {msg}")


# --------------------------------------------------------------------------------------------------
# torch <-> RlField helpers
# --------------------------------------------------------------------------------------------------
def field_of(t: torch.Tensor | None, layout: str | None = None) -> RlField:
    """View a 1-D / 2-D tensor as an RlField.

    ``layout`` = "soa": tensor is [C, N] (component-major, env innermost); "aos": tensor is [N, C...]
    (env-major, trailing dims flattened row-major); None: 1-D per-env tensor [N].
    """
    if t is None:
        return RlField(None, 0, 0)
    if not t.is_cuda:
        raise NativeError("device tensors only - the MDP step has no CPU path")
    if layout is None:
        if t.dim() != 1:
            raise ValueError("layout=None expects a 1-D tensor")
        return RlField(t.data_ptr(), t.stride(0), 0)
    if layout == "soa":
        if t.dim() == 1:
            return RlField(t.data_ptr(), t.stride(0), 0)
        if t.dim() != 2:
            raise ValueError("soa fields are [C, N]")
        return RlField(t.data_ptr(), t.stride(1), t.stride(0))
    if layout == "aos":
        if t.dim() == 1:
            return RlField(t.data_ptr(), t.stride(0), 0)
        flat = t.reshape(t.shape[0], -1)  # view when trailing dims are contiguous
        if flat.data_ptr() != t.data_ptr():
            raise ValueError("aos fields must have contiguous trailing dims")
        return RlField(flat.data_ptr(), flat.stride(0), flat.stride(1) if flat.shape[1] > 1 else 1)
    raise ValueError(layout)


def ptr_of(t: torch.Tensor | None) -> int | None:
    if t is None:
        return None
    if not t.is_cuda:
        raise NativeError("device tensors only - the MDP step has no CPU path")
    return t.data_ptr()
