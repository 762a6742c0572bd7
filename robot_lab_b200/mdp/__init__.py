"""MDP term functions with the reference's names and term protocol: ``func(env, **params) -> Tensor[N]``.

In the reference every term is a small eager-PyTorch function (V/mdp/rewards.py, V/mdp/observations.py, the
IsaacLab terms re-exported by V/mdp/__init__.py:11-20) that the managers call one by one. Here a term function
is (i) an *identifier* the spec compiler recognises and fuses into the single CUDA step kernel, and (ii) still a
callable with the same signature: calling it evaluates just that term on the GPU through ``rl_term_eval``
(reward terms) - the per-term entry point used by the unit-parity tests.

Nothing in here computes on the CPU; there is no fallback.
"""

from __future__ import annotations

from typing import Any, Callable

from .._native import DONE_TYPES, OBS_TYPES, REWARD_TYPES

_REGISTRY: dict[str, Callable] = {}


def _make(kind: str, name: str, type_name: str, ref: str, defaults: dict[str, Any] | None = None) -> Callable:
    table = {"reward": REWARD_TYPES, "obs": OBS_TYPES, "done": DONE_TYPES}[kind]
    type_id = table[type_name]

    def term(env, **params):
        merged = dict(defaults or {})
        merged.update(params)
        if kind == "reward":
            return env.reward_manager.evaluate_term(term, merged)
        if kind == "obs":
            return env.observation_manager.evaluate_term(term, merged)
        return env.termination_manager.evaluate_term(term, merged)

    term.__name__ = name
    term.__qualname__ = name
    term.__doc__ = f"{kind} term '{name}' - restates {ref}"
    term.rl_kind = kind
    term.rl_type_name = type_name
    term.rl_type_id = type_id
    term.rl_defaults = dict(defaults or {})
    _REGISTRY[name] = term
    return term


_R = "V/mdp/rewards.py"
_IL = "isaaclab.envs.mdp [IL]"

# --- reward terms owned by robot_lab (V/mdp/rewards.py) ---------------------------------------------
track_lin_vel_xy_exp = _make("reward", "track_lin_vel_xy_exp", "track_lin_vel_xy_exp", f"{_R}:22-35")
track_ang_vel_z_exp = _make("reward", "track_ang_vel_z_exp", "track_ang_vel_z_exp", f"{_R}:38-48")
track_lin_vel_xy_yaw_frame_exp = _make("reward", "track_lin_vel_xy_yaw_frame_exp", "track_lin_vel_xy_yaw_frame_exp", f"{_R}:51-66")
track_ang_vel_z_world_exp = _make("reward", "track_ang_vel_z_world_exp", "track_ang_vel_z_world_exp", f"{_R}:69-78")
joint_power = _make("reward", "joint_power", "joint_power", f"{_R}:81-90")
stand_still = _make("reward", "stand_still", "stand_still", f"{_R}:93-104", {"command_threshold": 0.06})
joint_pos_penalty = _make("reward", "joint_pos_penalty", "joint_pos_penalty", f"{_R}:107-129")
wheel_vel_penalty = _make("reward", "wheel_vel_penalty", "wheel_vel_penalty", f"{_R}:132-153")
GaitReward = _make("reward", "GaitReward", "feet_gait", f"{_R}:156-256")
joint_mirror = _make("reward", "joint_mirror", "joint_mirror", f"{_R}:259-278")
action_mirror = _make("reward", "action_mirror", "action_mirror", f"{_R}:281-303")
action_sync = _make("reward", "action_sync", "action_sync", f"{_R}:306-337")
feet_air_time = _make("reward", "feet_air_time", "feet_air_time", f"{_R}:340-360")
feet_air_time_positive_biped = _make("reward", "feet_air_time_positive_biped", "feet_air_time_positive_biped", f"{_R}:363-383")
feet_air_time_variance_penalty = _make("reward", "feet_air_time_variance_penalty", "feet_air_time_variance", f"{_R}:386-397")
feet_contact = _make("reward", "feet_contact", "feet_contact", f"{_R}:400-413")
feet_contact_without_cmd = _make("reward", "feet_contact_without_cmd", "feet_contact_without_cmd", f"{_R}:416-425")
feet_stumble = _make("reward", "feet_stumble", "feet_stumble", f"{_R}:428-436")
feet_distance_y_exp = _make("reward", "feet_distance_y_exp", "feet_distance_y_exp", f"{_R}:439-461")
feet_distance_xy_exp = _make("reward", "feet_distance_xy_exp", "feet_distance_xy_exp", f"{_R}:464-504")
feet_height = _make("reward", "feet_height", "feet_height", f"{_R}:507-524")
feet_height_body = _make("reward", "feet_height_body", "feet_height_body", f"{_R}:527-554")
feet_slide = _make("reward", "feet_slide", "feet_slide", f"{_R}:557-587")
upward = _make("reward", "upward", "upward", f"{_R}:608-613")
base_height_l2 = _make("reward", "base_height_l2", "base_height_l2", f"{_R}:616-644", {"sensor_cfg": None})
lin_vel_z_l2 = _make("reward", "lin_vel_z_l2", "lin_vel_z_l2", f"{_R}:647-653")
ang_vel_xy_l2 = _make("reward", "ang_vel_xy_l2", "ang_vel_xy_l2", f"{_R}:656-662")
undesired_contacts = _make("reward", "undesired_contacts", "undesired_contacts", f"{_R}:665-675")
flat_orientation_l2 = _make("reward", "flat_orientation_l2", "flat_orientation_l2", f"{_R}:678-687")

# --- reward terms owned by IsaacLab, called by the reference at V/velocity_env_cfg.py:379-523 -----------
is_terminated = _make("reward", "is_terminated", "is_terminated", f"{_IL} rewards.is_terminated")
joint_torques_l2 = _make("reward", "joint_torques_l2", "joint_torques_l2", f"{_IL} rewards.joint_torques_l2")
joint_vel_l2 = _make("reward", "joint_vel_l2", "joint_vel_l2", f"{_IL} rewards.joint_vel_l2")
joint_acc_l2 = _make("reward", "joint_acc_l2", "joint_acc_l2", f"{_IL} rewards.joint_acc_l2")
joint_deviation_l1 = _make("reward", "joint_deviation_l1", "joint_deviation_l1", f"{_IL} rewards.joint_deviation_l1")
joint_pos_limits = _make("reward", "joint_pos_limits", "joint_pos_limits", f"{_IL} rewards.joint_pos_limits")
joint_vel_limits = _make("reward", "joint_vel_limits", "joint_vel_limits", f"{_IL} rewards.joint_vel_limits")
action_rate_l2 = _make("reward", "action_rate_l2", "action_rate_l2", f"{_IL} rewards.action_rate_l2")
contact_forces = _make("reward", "contact_forces", "contact_forces", f"{_IL} rewards.contact_forces")

# --- observation terms -------------------------------------------------------------------------------
base_lin_vel = _make("obs", "base_lin_vel", "base_lin_vel", f"{_IL} observations.base_lin_vel")
base_ang_vel = _make("obs", "base_ang_vel", "base_ang_vel", f"{_IL} observations.base_ang_vel")
projected_gravity = _make("obs", "projected_gravity", "projected_gravity", f"{_IL} observations.projected_gravity")
generated_commands = _make("obs", "generated_commands", "generated_commands", f"{_IL} observations.generated_commands")
joint_pos_rel = _make("obs", "joint_pos_rel", "joint_pos_rel", f"{_IL} observations.joint_pos_rel")
joint_vel_rel = _make("obs", "joint_vel_rel", "joint_vel_rel", f"{_IL} observations.joint_vel_rel")
last_action = _make("obs", "last_action", "last_action", f"{_IL} observations.last_action")
height_scan = _make("obs", "height_scan", "height_scan", f"{_IL} observations.height_scan", {"offset": 0.5})
joint_pos_rel_without_wheel = _make("obs", "joint_pos_rel_without_wheel", "joint_pos_rel_without_wheel", "V/mdp/observations.py:17-27")
phase = _make("obs", "phase", "phase", "V/mdp/observations.py:30-35")

# --- termination terms ---------------------------------------------------------------------------------
time_out = _make("done", "time_out", "time_out", f"{_IL} terminations.time_out")
terrain_out_of_bounds = _make("done", "terrain_out_of_bounds", "terrain_out_of_bounds",
                              "isaaclab_tasks...velocity.mdp.terminations.terrain_out_of_bounds [IL]",
                              {"distance_buffer": 3.0})
illegal_contact = _make("done", "illegal_contact", "illegal_contact", f"{_IL} terminations.illegal_contact")


# --- event terms ------------------------------------------------------------------------------------------
# Not in the registry above: an event term is no term of the fused step. The env recognises this marker in
# ``cfg.events`` and runs it as ``rl_interval_push`` (stage 8 of the step); calling it directly is an error.
def push_by_setting_velocity(env, env_ids, velocity_range, asset_cfg=None):
    """push_by_setting_velocity [IL] (isaaclab.envs.mdp.events): root_vel_w[env_ids] += U(velocity_range). Runs on the
    device inside ``env.step()`` when configured as an interval event term (``ManagerBasedRLEnv`` / EventManager)."""
    raise NotImplementedError("push_by_setting_velocity runs inside env.step() as an interval event term (cfg.events)")


push_by_setting_velocity.rl_kind = "event"


def get(name: str) -> Callable:
    return _REGISTRY[name]


def all_terms() -> dict[str, Callable]:
    return dict(_REGISTRY)
