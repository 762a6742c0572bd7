"""Configuration classes of the manager-based MDP, with the names the reference's task files use.

The reference builds its tasks from IsaacLab cfg classes (``RewardTermCfg as RewTerm``, ``ObservationTermCfg
as ObsTerm``, ``ObservationGroupCfg``, ``TerminationTermCfg as DoneTerm``, ``SceneEntityCfg``,
``AdditiveUniformNoiseCfg as Unoise`` - V/velocity_env_cfg.py:15-27). Those classes live in IsaacLab, which is
not available here, so the same surface is provided natively: same field names, same meaning. They are plain
data - the spec compiler (``robot_lab_b200.spec``) turns a cfg tree into the flat ``RlStepSpec`` the CUDA
kernels consume.
"""

from __future__ import annotations

import copy
import re
from dataclasses import dataclass, field
from typing import Any, Callable, Sequence


# ------------------------------------------------------------------------------------------------
# name resolution (restates isaaclab.utils.string.resolve_matching_names [IL])
# ------------------------------------------------------------------------------------------------
def resolve_matching_names(
    keys: str | Sequence[str], names: Sequence[str], preserve_order: bool = False
) -> tuple[list[int], list[str]]:
    """Indices / names of ``names`` entries fully matched by one of the regex ``keys``.

    Without ``preserve_order`` the result follows the order of ``names``; with it, the order of ``keys``.
    A target matched by two keys, or a key that matches nothing, is an error (as upstream).
    """
    if isinstance(keys, str):
        keys = [keys]
    hits: list[tuple[int, int]] = []  # (key index, target index)
    matched_by: dict[int, str] = {}
    key_used = [False] * len(keys)
    for ti, target in enumerate(names):
        for ki, key in enumerate(keys):
            if re.fullmatch(key, target):
                if ti in matched_by:
                    raise ValueError(f"'{target}' matched by both '{matched_by[ti]}' and '{key}'")
                matched_by[ti] = key
                key_used[ki] = True
                hits.append((ki, ti))
    if not all(key_used):
        missing = [k for k, u in zip(keys, key_used) if not u]
        raise ValueError(f"no match for {missing} in {list(names)}")
    if preserve_order:
        hits.sort(key=lambda kt: kt[0])  # stable: ties keep target order
    ids = [ti for _, ti in hits]
    return ids, [names[i] for i in ids]


def resolve_matching_names_values(data: dict[str, Any], names: Sequence[str]) -> tuple[list[int], list[str], list[Any]]:
    """Per-name values from a ``{regex: value}`` dict (isaaclab.utils.string.resolve_matching_names_values [IL])."""
    ids, out_names, values = [], [], []
    used = {k: False for k in data}
    for ti, target in enumerate(names):
        found = None
        for key, val in data.items():
            if re.fullmatch(key, target):
                if found is not None:
                    raise ValueError(f"'{target}' matched by both '{found}' and '{key}'")
                found = key
                used[key] = True
                ids.append(ti)
                out_names.append(target)
                values.append(val)
    if not all(used.values()):
        raise ValueError(f"no match for {[k for k, u in used.items() if not u]} in {list(names)}")
    return ids, out_names, values


# ------------------------------------------------------------------------------------------------
# cfg classes
# ------------------------------------------------------------------------------------------------
@dataclass
class SceneEntityCfg:
    """Which joints / bodies of a scene entity a term acts on (isaaclab.managers.SceneEntityCfg [IL])."""

    name: str
    joint_names: str | list[str] | None = None
    body_names: str | list[str] | None = None
    preserve_order: bool = False
    # filled by resolve(): list of ints or slice(None) exactly like upstream
    joint_ids: Any = field(default_factory=lambda: slice(None))
    body_ids: Any = field(default_factory=lambda: slice(None))

    def resolve_joints(self, joint_names: Sequence[str]) -> list[int]:
        if self.joint_names is None:
            self.joint_ids = slice(None)
            return list(range(len(joint_names)))
        ids, _ = resolve_matching_names(self.joint_names, joint_names, self.preserve_order)
        self.joint_ids = slice(None) if ids == list(range(len(joint_names))) else ids
        return ids

    def resolve_bodies(self, body_names: Sequence[str]) -> list[int]:
        if self.body_names is None:
            self.body_ids = slice(None)
            return list(range(len(body_names)))
        ids, _ = resolve_matching_names(self.body_names, body_names, self.preserve_order)
        self.body_ids = slice(None) if ids == list(range(len(body_names))) else ids
        return ids

    def resolve(self, scene) -> None:
        """isaaclab.managers.SceneEntityCfg.resolve(scene) [IL]: fill joint_ids / body_ids against the named entity."""
        scene.resolve(self)


@dataclass
class AdditiveUniformNoiseCfg:
    n_min: float = -1.0
    n_max: float = 1.0


@dataclass
class RewardTermCfg:
    func: Callable
    weight: float
    params: dict[str, Any] = field(default_factory=dict)


@dataclass
class ObservationTermCfg:
    func: Callable
    params: dict[str, Any] = field(default_factory=dict)
    noise: AdditiveUniformNoiseCfg | None = None
    clip: tuple[float, float] | None = None
    scale: float | None = None


@dataclass
class TerminationTermCfg:
    func: Callable
    params: dict[str, Any] = field(default_factory=dict)
    time_out: bool = False


@dataclass
class EventTermCfg:
    """EventTermCfg [IL] (isaaclab.managers.EventTermCfg): ``func`` applied in ``mode`` ("startup" | "reset" |
    "interval"); interval terms fire every ``interval_range_s`` seconds, drawn per env unless ``is_global_time``."""

    func: Callable
    mode: str
    interval_range_s: tuple[float, float] | None = None
    is_global_time: bool = False
    params: dict[str, Any] = field(default_factory=dict)


class TermContainer:
    """An ordered bag of named terms; attribute order = insertion order (the managers iterate in it).

    Stands in for the ``@configclass`` classes of the reference (``RewardsCfg``, ``PolicyCfg`` ...): terms are
    attributes, ``None`` disables one, new attributes may be added later (V/velocity_env_cfg.py:411-417).
    """

    def __init__(self, **terms: Any):
        object.__setattr__(self, "_order", [])
        for k, v in terms.items():
            setattr(self, k, v)

    def __setattr__(self, key: str, value: Any) -> None:
        if not key.startswith("_") and key not in self._order:
            self._order.append(key)
        object.__setattr__(self, key, value)

    def items(self):
        return [(k, getattr(self, k)) for k in self._order]

    def active(self, kind: type | tuple[type, ...]):
        return [(k, v) for k, v in self.items() if v is not None and isinstance(v, kind)]

    def __deepcopy__(self, memo):
        new = type(self).__new__(type(self))
        object.__setattr__(new, "_order", list(self._order))
        for k, v in self.__dict__.items():
            if k != "_order":
                object.__setattr__(new, k, copy.deepcopy(v, memo))
        return new


class ObservationGroupCfg(TermContainer):
    """ObservationGroupCfg [IL]: terms in order + ``enable_corruption`` / ``concatenate_terms``."""

    def __init__(self, enable_corruption: bool = False, concatenate_terms: bool = True, **terms: Any):
        super().__init__(**terms)
        object.__setattr__(self, "enable_corruption", enable_corruption)
        object.__setattr__(self, "concatenate_terms", concatenate_terms)

    def __setattr__(self, key: str, value: Any) -> None:
        if key in ("enable_corruption", "concatenate_terms"):
            object.__setattr__(self, key, value)
        else:
            super().__setattr__(key, value)


@dataclass
class VelocityRanges:
    lin_vel_x: tuple[float, float] = (-1.0, 1.0)
    lin_vel_y: tuple[float, float] = (-1.0, 1.0)
    ang_vel_z: tuple[float, float] = (-1.0, 1.0)
    heading: tuple[float, float] | None = None


@dataclass
class UniformThresholdVelocityCommandCfg:
    """V/mdp/commands.py:88-92 over UniformVelocityCommandCfg [IL]; values at V/velocity_env_cfg.py:106-117."""

    asset_name: str = "robot"
    resampling_time_range: tuple[float, float] = (10.0, 10.0)
    rel_standing_envs: float = 0.0
    rel_heading_envs: float = 1.0
    heading_command: bool = False
    heading_control_stiffness: float = 1.0
    ranges: VelocityRanges = field(default_factory=VelocityRanges)
    small_command_threshold: float = 0.2  # V/mdp/commands.py:47 (hard-coded there)
    debug_vis: bool = False

    Ranges = VelocityRanges


@dataclass
class JointPositionActionCfg:
    """JointPositionActionCfg [IL] as used at V/velocity_env_cfg.py:124-126."""

    asset_name: str = "robot"
    joint_names: list[str] = field(default_factory=lambda: [".*"])
    scale: float | dict[str, float] = 1.0
    offset: float | dict[str, float] = 0.0
    use_default_offset: bool = True
    clip: dict[str, tuple[float, float]] | None = None
    preserve_order: bool = False


@dataclass
class JointVelocityActionCfg(JointPositionActionCfg):
    """JointVelocityActionCfg [IL]: the second action term of the wheeled robots (e.g.
    V/config/wheeled/unitree_go2w/rough_env_cfg.py:29-32, scale 5.0 at :102): same processing, the result is the joint
    VELOCITY target and ``use_default_offset`` takes the default joint velocity."""


@dataclass
class TerrainCfg:
    """The part of TerrainImporterCfg / TerrainGeneratorCfg [IL] the MDP terms read.

    Defaults are ROUGH_TERRAINS_CFG [IL]: 8 m tiles, 10 x 20 grid, 20 m border, sub-terrains without "pits"
    (SURVEY Appendix A), which makes V/mdp/utils.py:27-28 return None -> no pit restriction.
    """

    terrain_type: str = "generator"  # "generator" | "plane"
    size: tuple[float, float] = (8.0, 8.0)
    num_rows: int = 10
    num_cols: int = 20
    border_width: float = 20.0
    sub_terrains: tuple[str, ...] = (
        "pyramid_stairs", "pyramid_stairs_inv", "boxes", "random_rough", "hf_pyramid_slope", "hf_pyramid_slope_inv",
    )
    # SubTerrainBaseCfg.proportion of each entry above (ROUGH_TERRAINS_CFG [IL]); read by
    # _get_terrain_column_range (V/mdp/utils.py:16-41)
    proportions: tuple[float, ...] = (0.2, 0.2, 0.2, 0.2, 0.1, 0.1)
    horizontal_scale: float = 0.1   # height-field vertex spacing [IL]


@dataclass
class RayCasterCfg:
    """Grid height scanner (V/velocity_env_cfg.py:70-77): rays = (size/res + 1) per axis, x fastest."""

    resolution: float = 0.1
    size: tuple[float, float] = (1.6, 1.0)
    offset_z: float = 20.0

    @property
    def num_rays(self) -> int:
        nx = int(round(self.size[0] / self.resolution)) + 1
        ny = int(round(self.size[1] / self.resolution)) + 1
        return nx * ny


@dataclass
class ContactSensorCfg:
    history_length: int = 3
    track_air_time: bool = True
    force_threshold: float = 1.0


@dataclass
class ResetStateCfg:
    """The two mode="reset" events that write physical state (V/velocity_env_cfg.py:326-363): ``reset_root_state_uniform``
    pose / velocity ranges (x, y, z, roll, pitch, yaw; missing keys = (0, 0)) and ``reset_joints_by_scale`` ranges."""

    pose_range: dict = field(default_factory=lambda: {"x": (-0.5, 0.5), "y": (-0.5, 0.5), "yaw": (-3.14, 3.14)})
    velocity_range: dict = field(default_factory=lambda: {k: (-0.5, 0.5) for k in ("x", "y", "z", "roll", "pitch", "yaw")})
    joint_position_range: tuple = (1.0, 1.0)
    joint_velocity_range: tuple = (0.0, 0.0)

    @staticmethod
    def go2_rough() -> "ResetStateCfg":
        """GO2/rough_env_cfg.py:56-73."""
        return ResetStateCfg(pose_range={"x": (-0.5, 0.5), "y": (-0.5, 0.5), "z": (0.0, 0.2), "roll": (-3.14, 3.14),
                                         "pitch": (-3.14, 3.14), "yaw": (-3.14, 3.14)})
