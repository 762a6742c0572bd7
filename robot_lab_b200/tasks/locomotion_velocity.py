"""Velocity-tracking locomotion task definition (the *spec* the fused kernel is parameterised from).

Re-expresses, table-driven and without IsaacLab imports, what the reference declares in
V/velocity_env_cfg.py: scene sensors (:70-86), command (:106-117), action (:124-126), the policy and critic
observation groups (:134-254), the reward-term catalogue with every weight at 0 (:379-644), terminations
(:652-664), decimation / dt / episode length (:714-717) and ``disable_zero_weight_rewards`` (:737-743).
Per-robot files (``unitree.py`` next to this one) then set weights and names exactly like the reference's
``rough_env_cfg.py`` / ``flat_env_cfg.py`` override chains do.

Events (startup / reset randomisation) and curricula are physics-side or host-side pieces outside the MDP step
(SURVEY.md section 2 rows 5-6); they are not represented here, with one exception: the interval push
``randomize_push_robot`` (V/velocity_env_cfg.py:366-371), stage 8 of the env step. ``cfg.events.randomize_push_robot``
is None (off) by default, so every task keeps the step without pushes; ``push_robot_event_term()`` returns the
reference's term, which the reference has on by default.
"""

from __future__ import annotations

import math
from dataclasses import dataclass, field

from .. import mdp
from ..assets import RobotAsset
from ..cfg import (
    AdditiveUniformNoiseCfg as Unoise,
    ContactSensorCfg,
    EventTermCfg as EventTerm,
    JointPositionActionCfg,
    ObservationGroupCfg as ObsGroup,
    ObservationTermCfg as ObsTerm,
    RayCasterCfg,
    RewardTermCfg as RewTerm,
    SceneEntityCfg,
    TermContainer,
    TerminationTermCfg as DoneTerm,
    TerrainCfg,
    UniformThresholdVelocityCommandCfg,
)
from ..spec import SceneLayout


@dataclass
class SceneCfg:
    """MySceneCfg (V/velocity_env_cfg.py:43-94), reduced to what the MDP terms read."""

    num_envs: int = 4096
    env_spacing: float = 2.5
    robot: RobotAsset | None = None
    terrain: TerrainCfg = field(default_factory=TerrainCfg)
    height_scanner: RayCasterCfg | None = field(default_factory=RayCasterCfg)
    contact_forces: ContactSensorCfg = field(default_factory=ContactSensorCfg)
    # "full": every body in every body-indexed tensor (IsaacLab-shaped); "compact": only bodies some term reads
    body_tensors: str = "compact"
    foot_body_regex: str = ".*_foot"

    def make_layout(self) -> SceneLayout:
        rays = self.height_scanner.num_rays if self.height_scanner is not None else 0
        return SceneLayout.full(self.robot, self.terrain, rays, self.contact_forces.history_length)


@dataclass
class SimCfg:
    dt: float = 0.005
    device: str = "cuda:0"


_CMD = {"command_name": "base_velocity"}


def _robot(**kw) -> SceneEntityCfg:
    return SceneEntityCfg("robot", **kw)


def _contacts(**kw) -> SceneEntityCfg:
    return SceneEntityCfg("contact_forces", **kw)


def _reward_catalogue() -> TermContainer:
    """All reward terms the reference declares, in its order, weight 0 (V/velocity_env_cfg.py:379-644)."""
    std_quarter = math.sqrt(0.25)
    rows = [
        ("is_terminated", mdp.is_terminated, {}),
        ("lin_vel_z_l2", mdp.lin_vel_z_l2, {}),
        ("ang_vel_xy_l2", mdp.ang_vel_xy_l2, {}),
        ("flat_orientation_l2", mdp.flat_orientation_l2, {}),
        ("base_height_l2", mdp.base_height_l2,
         {"asset_cfg": _robot(body_names=""), "sensor_cfg": SceneEntityCfg("height_scanner_base"), "target_height": 0.0}),
        ("joint_torques_l2", mdp.joint_torques_l2, {"asset_cfg": _robot(joint_names=".*")}),
        ("joint_vel_l2", mdp.joint_vel_l2, {"asset_cfg": _robot(joint_names=".*")}),
        ("joint_acc_l2", mdp.joint_acc_l2, {"asset_cfg": _robot(joint_names=".*")}),
        ("joint_pos_limits", mdp.joint_pos_limits, {"asset_cfg": _robot(joint_names=".*")}),
        ("joint_vel_limits", mdp.joint_vel_limits, {"asset_cfg": _robot(joint_names=".*"), "soft_ratio": 1.0}),
        ("joint_power", mdp.joint_power, {"asset_cfg": _robot(joint_names=".*")}),
        ("stand_still", mdp.stand_still, {**_CMD, "command_threshold": 0.1, "asset_cfg": _robot(joint_names=".*")}),
        ("joint_pos_penalty", mdp.joint_pos_penalty,
         {**_CMD, "asset_cfg": _robot(joint_names=".*"), "stand_still_scale": 5.0, "velocity_threshold": 0.5,
          "command_threshold": 0.1}),
        ("wheel_vel_penalty", mdp.wheel_vel_penalty,
         {"asset_cfg": _robot(joint_names=""), "sensor_cfg": _contacts(body_names=""), **_CMD,
          "velocity_threshold": 0.5, "command_threshold": 0.1}),
        ("joint_mirror", mdp.joint_mirror, {"asset_cfg": _robot(), "mirror_joints": [["FR.*", "RL.*"], ["FL.*", "RR.*"]]}),
        ("action_mirror", mdp.action_mirror, {"asset_cfg": _robot(), "mirror_joints": [["FR.*", "RL.*"], ["FL.*", "RR.*"]]}),
        ("action_sync", mdp.action_sync,
         {"asset_cfg": _robot(),
          "joint_groups": [[f"{leg}_{part}_joint" for leg in ("FR", "FL", "RL", "RR")] for part in ("hip", "thigh", "calf")]}),
        ("action_rate_l2", mdp.action_rate_l2, {}),
        ("undesired_contacts", mdp.undesired_contacts, {"sensor_cfg": _contacts(body_names=""), "threshold": 1.0}),
        ("contact_forces", mdp.contact_forces, {"sensor_cfg": _contacts(body_names=""), "threshold": 100.0}),
        ("track_lin_vel_xy_exp", mdp.track_lin_vel_xy_exp, {**_CMD, "std": std_quarter}),
        ("track_ang_vel_z_exp", mdp.track_ang_vel_z_exp, {**_CMD, "std": std_quarter}),
        ("feet_air_time", mdp.feet_air_time, {**_CMD, "threshold": 0.5, "sensor_cfg": _contacts(body_names="")}),
        ("feet_air_time_variance", mdp.feet_air_time_variance_penalty, {"sensor_cfg": _contacts(body_names="")}),
        ("feet_gait", mdp.GaitReward,
         {"std": math.sqrt(0.5), **_CMD, "max_err": 0.2, "velocity_threshold": 0.5, "command_threshold": 0.1,
          "synced_feet_pair_names": (("", ""), ("", "")), "asset_cfg": _robot(), "sensor_cfg": _contacts()}),
        ("feet_contact", mdp.feet_contact, {"sensor_cfg": _contacts(body_names=""), **_CMD, "expect_contact_num": 2}),
        ("feet_contact_without_cmd", mdp.feet_contact_without_cmd, {"sensor_cfg": _contacts(body_names=""), **_CMD}),
        ("feet_stumble", mdp.feet_stumble, {"sensor_cfg": _contacts(body_names="")}),
        ("feet_slide", mdp.feet_slide, {"sensor_cfg": _contacts(body_names=""), "asset_cfg": _robot(body_names="")}),
        ("feet_height", mdp.feet_height, {"asset_cfg": _robot(body_names=""), "tanh_mult": 2.0, "target_height": 0.05, **_CMD}),
        ("feet_height_body", mdp.feet_height_body, {"asset_cfg": _robot(body_names=""), "tanh_mult": 2.0, "target_height": -0.3, **_CMD}),
        ("feet_distance_y_exp", mdp.feet_distance_y_exp, {"std": std_quarter, "asset_cfg": _robot(body_names=""), "stance_width": float}),
        ("upward", mdp.upward, {}),
    ]
    # body_lin_acc_l2 and applied_torque_limits (V/velocity_env_cfg.py:394-398,501-505) need state the MDP-step
    # boundary does not carry (body accelerations, pre-clip torques); they have weight 0 in every in-scope task.
    bag = TermContainer()
    for name, func, params in rows:
        setattr(bag, name, RewTerm(func=func, weight=0.0, params=params))
    return bag


def _obs_group(corrupt: bool) -> ObsGroup:
    """PolicyCfg (noise on) / CriticCfg (noise off): V/velocity_env_cfg.py:134-254."""
    noise = (lambda lo, hi: Unoise(n_min=lo, n_max=hi)) if corrupt else (lambda lo, hi: None)
    c100 = (-100.0, 100.0)
    g = ObsGroup(enable_corruption=corrupt, concatenate_terms=True)
    g.base_lin_vel = ObsTerm(func=mdp.base_lin_vel, noise=noise(-0.1, 0.1), clip=c100, scale=1.0)
    g.base_ang_vel = ObsTerm(func=mdp.base_ang_vel, noise=noise(-0.2, 0.2), clip=c100, scale=1.0)
    g.projected_gravity = ObsTerm(func=mdp.projected_gravity, noise=noise(-0.05, 0.05), clip=c100, scale=1.0)
    g.velocity_commands = ObsTerm(func=mdp.generated_commands, params=dict(_CMD), clip=c100, scale=1.0)
    g.joint_pos = ObsTerm(func=mdp.joint_pos_rel, params={"asset_cfg": _robot(joint_names=".*", preserve_order=True)},
                          noise=noise(-0.01, 0.01), clip=c100, scale=1.0)
    g.joint_vel = ObsTerm(func=mdp.joint_vel_rel, params={"asset_cfg": _robot(joint_names=".*", preserve_order=True)},
                          noise=noise(-1.5, 1.5), clip=c100, scale=1.0)
    g.actions = ObsTerm(func=mdp.last_action, clip=c100, scale=1.0)
    g.height_scan = ObsTerm(func=mdp.height_scan, params={"sensor_cfg": SceneEntityCfg("height_scanner")},
                            noise=noise(-0.1, 0.1), clip=(-1.0, 1.0), scale=1.0)
    return g


def push_robot_event_term(interval_range_s: tuple[float, float] = (10.0, 15.0),
                          velocity_range: dict | None = None) -> EventTerm:
    """The reference's ``randomize_push_robot`` (V/velocity_env_cfg.py:366-371): push_by_setting_velocity every 10 to
    15 s per env. The term, its function and the interval are the reference's (SURVEY.md section 3.2, stage 8); the
    x / y range of +-0.5 m/s is the value of the IsaacLab locomotion velocity template that file follows
    (isaaclab_tasks .../locomotion/velocity/velocity_env_cfg.py, ``push_robot``), not read from the reference itself."""
    if velocity_range is None:
        velocity_range = {"x": (-0.5, 0.5), "y": (-0.5, 0.5)}
    return EventTerm(func=mdp.push_by_setting_velocity, mode="interval", interval_range_s=interval_range_s,
                     params={"velocity_range": velocity_range})


class LocomotionVelocityRoughEnvCfg:
    """Base task cfg (V/velocity_env_cfg.py:695-743)."""

    task_name = "LocomotionVelocityRough"

    def __init__(self) -> None:
        self.seed = 42
        self.scene = SceneCfg()
        self.sim = SimCfg()
        self.observations = TermContainer(policy=_obs_group(True), critic=_obs_group(False))
        self.actions = TermContainer(joint_pos=JointPositionActionCfg(
            asset_name="robot", joint_names=[".*"], scale=0.5, use_default_offset=True, clip=None, preserve_order=True))
        self.commands = TermContainer(base_velocity=UniformThresholdVelocityCommandCfg(
            asset_name="robot", resampling_time_range=(10.0, 10.0), rel_standing_envs=0.02, rel_heading_envs=1.0,
            heading_command=True, heading_control_stiffness=0.5, debug_vis=True,
            ranges=UniformThresholdVelocityCommandCfg.Ranges(
                lin_vel_x=(-1.0, 1.0), lin_vel_y=(-1.0, 1.0), ang_vel_z=(-1.0, 1.0), heading=(-math.pi, math.pi))))
        self.rewards = _reward_catalogue()
        self.terminations = TermContainer(
            time_out=DoneTerm(func=mdp.time_out, time_out=True),
            terrain_out_of_bounds=DoneTerm(func=mdp.terrain_out_of_bounds,
                                           params={"asset_cfg": _robot(), "distance_buffer": 3.0}, time_out=True),
            illegal_contact=DoneTerm(func=mdp.illegal_contact,
                                     params={"sensor_cfg": _contacts(body_names=""), "threshold": 1.0}),
        )
        # interval events: off by default (the reference enables randomize_push_robot; push_robot_event_term() is it)
        self.events = TermContainer(randomize_push_robot=None)
        self.decimation = 4
        self.episode_length_s = 20.0
        self.sim.dt = 0.005

    # -- helpers mirroring the reference cfg methods --------------------------------------------------
    def create_joint_deviation_l1_rewterm(self, attr_name: str, weight: float, joint_names_pattern) -> None:
        """V/velocity_env_cfg.py:411-417."""
        setattr(self.rewards, attr_name, RewTerm(func=mdp.joint_deviation_l1, weight=weight,
                                                 params={"asset_cfg": _robot(joint_names=joint_names_pattern)}))

    def disable_zero_weight_rewards(self) -> None:
        """If the weight of rewards is 0, set rewards to None (V/velocity_env_cfg.py:737-743)."""
        for name, term in self.rewards.items():
            if isinstance(term, RewTerm) and term.weight == 0:
                setattr(self.rewards, name, None)

    @property
    def step_dt(self) -> float:
        return self.sim.dt * self.decimation

    @property
    def max_episode_length(self) -> int:
        return math.ceil(self.episode_length_s / self.step_dt)
