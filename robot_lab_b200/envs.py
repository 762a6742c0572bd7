"""``ManagerBasedRLEnv`` + managers + ``RslRlVecEnvWrapper`` with the API surface the reference's scripts consume.

What the reference relies on (SURVEY.md 8(b).3; scripts/reinforcement_learning/rsl_rl/train.py:177-224,
play.py:175-248, scripts/tools/zero_agent.py:56-70): ``gym.make(id, cfg=env_cfg)`` -> env with ``.unwrapped``,
``.num_envs``, ``.device``, ``.observation_space`` / ``.action_space``, ``.reset()``, ``.step(a) -> (obs_dict{"policy",
"critic"}, rew[N], terminated[N] bool, truncated[N] bool, extras{"log": ...})``, ``.close()``; the wrapper adds
``num_actions``, ``max_episode_length``, ``episode_length_buf`` (get/set), ``get_observations()``, ``step(actions) ->
(obs, rew, dones long, extras with "time_outs")``. Term functions read ``env.scene[...]``, ``env.command_manager``,
``env.action_manager`` (SURVEY.md 8(b).2) - those attributes exist here too, backed by the device buffers.

In IsaacLab each manager loops over its terms in Python. Here ``env.step()`` is three CUDA launches
(``rl_process_action`` -> state provider -> ``rl_step`` -> provider reset -> post-reset launch), plus the interval push
and a re-observation of the pushed envs when ``cfg.events`` enables it; the manager
objects are views onto the buffers those launches fill, plus per-manager ``compute()`` entry points that run just
their phase of the kernel. There is no CPU implementation behind any of this.

Physics is not part of this tier: a ``StateProvider`` fills the state buffers each step. ``SyntheticStateProvider``
(the default) draws fresh synthetic state on the device; a simulator integration implements the same two methods.
"""

from __future__ import annotations

import math
from typing import Any

import torch

from . import _native as nat
from .cfg import RewardTermCfg
from .engine import MdpStepEngine
from .spec import StepSpec, compact_layout, compile_reward_term, compile_step_spec
from .state import StateBuffers
from .synthetic import make_state

import os as _os

_NVTX = _os.environ.get("RL_MDP_NVTX", "0") == "1"

try:  # optional: real gymnasium spaces / registration when the package exists
    import gymnasium as gym  # type: ignore
except Exception:  # pragma: no cover - not installed in the build image
    gym = None

try:
    from tensordict import TensorDict  # type: ignore
except Exception:  # pragma: no cover
    TensorDict = None


class Box:
    """Minimal stand-in for ``gymnasium.spaces.Box`` (shape / dtype / bounds) when gymnasium is absent."""

    def __init__(self, low: float, high: float, shape: tuple[int, ...], dtype=torch.float32):
        self.low, self.high, self.shape, self.dtype = low, high, tuple(shape), dtype

    def __repr__(self):
        return f"Box({self.low}, {self.high}, {self.shape})"


# --------------------------------------------------------------------------------------------------
# state providers (the physics / sensor side of the boundary)
# --------------------------------------------------------------------------------------------------
class StateProvider:
    """Producer of the per-step state buffers (root / joint state, contact history, timers, feet kinematics, rays)."""

    def advance(self, env: "ManagerBasedRLEnv") -> None:  # after process_action, before the fused step
        raise NotImplementedError

    def reset(self, env: "ManagerBasedRLEnv", env_ids: torch.Tensor, n_ids: torch.Tensor) -> None:
        """Write post-reset physical state for ``env_ids[: n_ids]`` (device tensors; no host sync required)."""


class SyntheticStateProvider(StateProvider):
    """Rotates over a few pre-generated synthetic state sets (device copies) - the benchmark's producer."""

    def __init__(self, spec: StepSpec, num_envs: int, device, num_sets: int = 4, seed: int = 1234, rank: int = 0):
        self.sets = []
        for i in range(num_sets):
            st = make_state(spec, num_envs, seed=seed + 1000 * i, rank=rank)
            self.sets.append({k: v for k, v in st.items() if k in nat._STATE_FIELDS})
        self.i = 0
        self._staged = None

    def advance(self, env):
        st = self.sets[self.i % len(self.sets)]
        self.i += 1
        for name, val in st.items():
            env.buffers._to_device(name, val)

    def reset(self, env, env_ids, n_ids):
        return  # synthetic state has no notion of a physical reset


class ResetEventStateProvider(SyntheticStateProvider):
    """Synthetic producer whose ``reset`` applies the reference's mode="reset" state events on the device
    (``reset_root_state_uniform`` V/mdp/events.py:205-271 + ``reset_joints_by_scale`` [IL]) through
    ``rl_reset_scene_state`` - the post-reset root / joint state the observation launch then reads."""

    def __init__(self, spec: StepSpec, num_envs: int, device, reset_cfg=None, env_origins: torch.Tensor | None = None, **kw):
        super().__init__(spec, num_envs, device, **kw)
        from .cfg import ResetStateCfg

        self.reset_cfg = reset_cfg if reset_cfg is not None else ResetStateCfg()
        self.env_origins = env_origins if env_origins is not None else torch.zeros(num_envs, 3, device=device)

    def reset(self, env, env_ids, n_ids):
        env.engine.reset_scene_state(env.buffers, self.reset_cfg, self.env_origins, env_ids=env_ids, n_env_ids=n_ids,
                                     seed=env.seed, env_id_offset=env.rank * env.num_envs, use_step_counter=True)


class SensorChainStateProvider(ResetEventStateProvider):
    """Synthetic root / joint / contact-force state, with everything the library can derive from it computed on the
    device in IsaacLab's order for every physics sub-step (``decimation`` of them, V/velocity_env_cfg.py:714):
    ``rl_actuator_step`` (joint target -> applied torque, SURVEY.md 8(f) row 3), ``rl_contact_sensor_update`` (force
    history + air / contact timers, row 1) and - once per env step, on the final pose - ``rl_height_scan_cast`` (the
    height scanner over a height field, row 4). ``reset`` is ``rl_reset_scene_state`` (row 2)."""

    def __init__(self, spec: StepSpec, num_envs: int, device, height_field=None, decimation: int = 4,
                 physics_dt: float = 0.005, **kw):
        super().__init__(spec, num_envs, device, **kw)
        self.height_field, self.decimation, self.physics_dt = height_field, decimation, physics_dt
        self.forces = [st["net_forces_w_history"][:, 0].contiguous().to(device) for st in self.sets]
        derived = ("applied_torque", "net_forces_w_history", "current_air_time", "last_air_time", "current_contact_time",
                   "last_contact_time") + (("ray_hits_z", "ray_sensor_pos_z") if height_field is not None else ())
        for st in self.sets:
            for k in derived:
                st.pop(k, None)
        self.substep = 0

    def advance(self, env):
        i = self.i % len(self.sets)
        super().advance(env)
        b, eng = env.buffers, env.engine
        # ring-slot writes move no data, but feet_stumble reads history slot 0 as "the newest sample" (net_forces_w,
        # V/mdp/rewards.py:431-434): a spec with that term active keeps IsaacLab's rolling history
        ring = not any(r.type_name == "feet_stumble" and r.weight != 0.0 for r in env.spec.rewards)
        for _ in range(self.decimation):
            eng.actuator_step(b)
            eng.contact_sensor_update(b, self.forces[i], self.physics_dt, ring_slot=(self.substep % env.spec.T) if ring else -1)
            self.substep += 1
        if self.height_field is not None and env.spec.R > 0:
            eng.height_scan_cast(b, self.height_field)


class ReplayStateProvider(StateProvider):
    """Feeds a fixed list of logical state dicts, one per step (tests: the oracle replays the same list)."""

    def __init__(self, states: list[dict]):
        self.states, self.i = states, 0

    def advance(self, env):
        st = self.states[self.i]
        self.i += 1
        for name in nat._STATE_FIELDS:
            env.buffers._to_device(name, st[name])


# --------------------------------------------------------------------------------------------------
# scene views: what Python term functions read through ``env`` (SURVEY.md 8(b).2). Raw fields are views of the device
# buffers; derived fields (ArticulationData properties [IL]) are device tensors filled lazily by ``rl_derived_views``,
# once per state version (the env bumps the version whenever a provider or a launch changes the physical state).
# --------------------------------------------------------------------------------------------------
class _ArticulationData:
    _RAW = ("root_pos_w", "root_quat_w", "root_lin_vel_w", "root_ang_vel_w", "joint_pos", "joint_vel", "joint_acc",
            "applied_torque", "body_pos_w", "body_lin_vel_w")
    _ALIAS = {"root_link_pos_w": "root_pos_w", "root_link_quat_w": "root_quat_w", "body_link_pos_w": "body_pos_w",
              "root_com_lin_vel_w": "root_lin_vel_w", "root_com_ang_vel_w": "root_ang_vel_w",
              "body_com_lin_vel_w": "body_lin_vel_w", "joint_pos_target": "joint_target"}
    _DERIVED = {"projected_gravity_b": 0, "root_lin_vel_b": 1, "root_ang_vel_b": 2, "root_com_lin_vel_b": 1,
                "root_com_ang_vel_b": 2, "root_link_lin_vel_b": 1, "root_link_ang_vel_b": 2}

    def __init__(self, env):
        self._env = env
        n, dev = env.num_envs, env.device
        self._vec = torch.zeros(3, n, 3, device=dev)       # projected_gravity_b, root_lin_vel_b, root_ang_vel_b
        self._heading = torch.zeros(n, device=dev)
        self._version = -1
        asset = env.spec.layout.asset
        f32 = dict(dtype=torch.float32, device=dev)
        self.default_joint_pos = torch.tensor(asset.default_joint_pos(), **f32).unsqueeze(0).expand(n, -1)
        self.default_joint_vel = torch.tensor(asset.default_joint_vel(), **f32).unsqueeze(0).expand(n, -1)
        self.soft_joint_pos_limits = torch.tensor(asset.soft_joint_pos_limits(), **f32).unsqueeze(0).expand(n, -1, -1)
        self.soft_joint_vel_limits = torch.tensor(asset.joint_vel_limits(), **f32).unsqueeze(0).expand(n, -1)
        root = [0.0, 0.0, asset.init_root_height, 1.0, 0.0, 0.0, 0.0] + [0.0] * 6
        self.default_root_state = torch.tensor(root, **f32).unsqueeze(0).expand(n, -1)

    def _refresh(self):
        env = self._env
        if self._version == env._state_version:
            return
        b = env.buffers
        st = b.state_view()
        vec = [nat.RlField(self._vec[i].data_ptr(), 3, 1) for i in range(3)]
        head = nat.RlField(self._heading.data_ptr(), 1, 1)
        import ctypes as C

        nat.check(env.engine.lib.rl_derived_views(env.engine._ctx, b.N, C.byref(st), C.byref(vec[0]), C.byref(vec[1]),
                                                  C.byref(vec[2]), C.byref(head), env.engine._stream()))
        self._version = env._state_version

    def __getattr__(self, name):
        cls = type(self)
        if name in cls._RAW:
            return self._env.buffers.logical(name)
        if name in cls._ALIAS:
            return self._env.buffers.logical(cls._ALIAS[name])
        if name in cls._DERIVED:
            self._refresh()
            return self._vec[cls._DERIVED[name]]
        if name == "heading_w":
            self._refresh()
            return self._heading
        raise AttributeError(f"ArticulationData has no field '{name}' on this env surface")


class _Articulation:
    def __init__(self, env):
        self._env = env
        self.data = _ArticulationData(env)
        asset = env.spec.layout.asset
        self.joint_names, self.body_names = list(asset.joint_names), list(env.spec.layout.asset_body_names)
        self.num_joints, self.num_bodies = asset.num_joints, len(self.body_names)

    def find_joints(self, name_keys, preserve_order: bool = False):
        from .cfg import resolve_matching_names

        return resolve_matching_names(name_keys, self.joint_names, preserve_order)

    def find_bodies(self, name_keys, preserve_order: bool = False):
        from .cfg import resolve_matching_names

        return resolve_matching_names(name_keys, self.body_names, preserve_order)


class _ContactSensorData:
    _RAW = ("net_forces_w_history", "current_air_time", "last_air_time", "current_contact_time", "last_contact_time")

    def __init__(self, env):
        self._env = env

    def __getattr__(self, name):
        if name in type(self)._RAW:
            return self._env.buffers.logical(name)
        if name == "net_forces_w":   # the newest history sample (slot 0 unless the provider writes ring slots)
            slot = int(getattr(self._env.state_provider, "newest_history_slot", 0))
            return self._env.buffers.logical("net_forces_w_history")[:, slot]
        raise AttributeError(f"ContactSensorData has no field '{name}' on this env surface")


class _ContactSensor:
    """ContactSensor [IL] surface. With the compact body layout the timer tensors hold the timer bodies only and the
    force history its own body list; ``body_tensors="full"`` gives every tensor every body, IsaacLab-style, so that one
    ``SceneEntityCfg.body_ids`` indexes them all."""

    def __init__(self, env):
        self._env = env
        self.data = _ContactSensorData(env)
        self.body_names = list(env.spec.layout.time_body_names)
        self.history_body_names = list(env.spec.layout.hist_body_names)

    def find_bodies(self, name_keys, preserve_order: bool = False):
        from .cfg import resolve_matching_names

        return resolve_matching_names(name_keys, self.body_names, preserve_order)

    def compute_first_contact(self, dt: float, abs_tol: float = 1.0e-8) -> torch.Tensor:
        t = self.data.current_contact_time
        return (t > 0.0) & (t < (dt + abs_tol))

    def compute_first_air(self, dt: float, abs_tol: float = 1.0e-8) -> torch.Tensor:
        t = self.data.current_air_time
        return (t > 0.0) & (t < (dt + abs_tol))


class _RayCasterData:
    def __init__(self, env):
        self._env = env
        from . import terrain as _terrain
        from .cfg import RayCasterCfg

        self._starts = _terrain.grid_pattern_ray_starts(RayCasterCfg()).to(env.device)   # [R, 3] sensor frame

    @property
    def pos_w(self) -> torch.Tensor:
        b = self._env.buffers
        pos = b.logical("root_pos_w")
        return torch.stack([pos[:, 0], pos[:, 1], b.logical("ray_sensor_pos_z")], dim=-1)

    @property
    def ray_hits_w(self) -> torch.Tensor:
        """[N, R, 3]: x, y of the yaw-aligned grid pattern under the sensor, z = the hit heights the step consumes."""
        b = self._env.buffers
        heading = self._env.scene["robot"].data.heading_w
        c, s = torch.cos(heading)[:, None], torch.sin(heading)[:, None]
        sx, sy = self._starts[None, :, 0], self._starts[None, :, 1]
        pos = b.logical("root_pos_w")
        x = pos[:, 0:1] + c * sx - s * sy
        y = pos[:, 1:2] + s * sx + c * sy
        return torch.stack([x, y, b.logical("ray_hits_z")], dim=-1)


class _RayCaster:
    """The grid height scanner (V/velocity_env_cfg.py:70-77) as terms see it: ``data.pos_w``, ``data.ray_hits_w``."""

    def __init__(self, env):
        self.data = _RayCasterData(env)


class _TerrainGeneratorCfgView:
    """The attributes of TerrainGeneratorCfg [IL] the reference reads (V/mdp/utils.py:16-41)."""

    class _Sub:
        def __init__(self, proportion):
            self.proportion = proportion

    def __init__(self, cfg):
        self.num_rows, self.num_cols, self.size, self.border_width = cfg.num_rows, cfg.num_cols, cfg.size, cfg.border_width
        self.sub_terrains = {name: self._Sub(p) for name, p in zip(cfg.sub_terrains, cfg.proportions)}


class _TerrainCfgView:
    def __init__(self, cfg):
        self.terrain_type = cfg.terrain_type
        self.terrain_generator = _TerrainGeneratorCfgView(cfg) if cfg.terrain_type == "generator" else None


class _Terrain:
    """TerrainImporter [IL] surface: ``cfg.terrain_type``, ``cfg.terrain_generator``, ``terrain_origins`` [rows, cols, 3],
    ``terrain_types`` [N] (column of every env's cell), ``env_origins`` [N, 3] (V/mdp/utils.py:42-127, events.py:240,257)."""

    def __init__(self, env, terrain_origins=None, terrain_types=None, env_origins=None):
        from . import terrain as _terrain

        tcfg = env.spec.layout.terrain
        self.cfg = _TerrainCfgView(tcfg)
        n, dev = env.num_envs, env.device
        if tcfg.terrain_type == "generator":
            self.terrain_origins = (terrain_origins if terrain_origins is not None else _terrain.grid_origins(tcfg)).to(dev)
            if terrain_types is None:   # TerrainImporter._compute_env_origins_curriculum [IL]: envs dealt round-robin to the columns
                terrain_types = torch.div(torch.arange(n), max(n / tcfg.num_cols, 1.0), rounding_mode="floor").to(torch.long)
            self.terrain_types = terrain_types.to(dev)
            if env_origins is None:
                env_origins = self.terrain_origins[0, self.terrain_types.clamp(max=tcfg.num_cols - 1)]
        else:
            self.terrain_origins, self.terrain_types = None, None
            if env_origins is None:
                env_origins = torch.zeros(n, 3)
        self.env_origins = env_origins.to(dev, torch.float32)


class _Scene(dict):
    def __init__(self, env, **terrain_kw):
        super().__init__(robot=_Articulation(env))
        self.sensors = {"contact_forces": _ContactSensor(env)}
        self["contact_forces"] = self.sensors["contact_forces"]
        if env.spec.R > 0:
            self.sensors["height_scanner"] = _RayCaster(env)
            self["height_scanner"] = self.sensors["height_scanner"]
        self.terrain = _Terrain(env, **terrain_kw)
        self.env_origins = self.terrain.env_origins
        self.num_envs = env.num_envs
        self.cfg = env.cfg.scene

    def resolve(self, entity_cfg):
        """``SceneEntityCfg.resolve(scene)`` [IL]: fill ``joint_ids`` / ``body_ids`` against this scene's entity."""
        ent = self[entity_cfg.name]
        if hasattr(ent, "joint_names"):
            entity_cfg.resolve_joints(ent.joint_names)
        entity_cfg.resolve_bodies(ent.body_names)
        return entity_cfg


# --------------------------------------------------------------------------------------------------
# managers
# --------------------------------------------------------------------------------------------------
class _ManagerBase:
    def __init__(self, env: "ManagerBasedRLEnv"):
        self._env = env

    @property
    def num_envs(self):
        return self._env.num_envs

    @property
    def device(self):
        return self._env.device


class ActionManager(_ManagerBase):
    @property
    def action(self) -> torch.Tensor:
        return self._env.buffers.logical("action")

    @property
    def prev_action(self) -> torch.Tensor:
        return self._env.buffers.logical("prev_action")

    @property
    def total_action_dim(self) -> int:
        return self._env.spec.A

    @property
    def processed_actions(self) -> torch.Tensor:
        """Joint position targets in native joint order (what ``apply_action`` would hand to the articulation)."""
        return self._env.buffers.logical("joint_target")

    def process_action(self, action: torch.Tensor) -> None:
        env = self._env
        if action.shape != (env.num_envs, env.spec.A):
            raise ValueError(f"Invalid action shape, expected: {(env.num_envs, env.spec.A)}, received: {tuple(action.shape)}.")
        if action.dtype == torch.float32 and action.device == env.device:
            env.engine.process_action(env.buffers, new_action=action)   # read in place: any strides, no staging copy
        else:
            env.buffers.t["new_action"].copy_(action.to(env.device, torch.float32))
            env.engine.process_action(env.buffers)


class RewardManager(_ManagerBase):
    def __init__(self, env):
        super().__init__(env)
        self.active_terms = [t.name for t in env.spec.rewards]
        self._term_cfgs = dict(env.cfg.rewards.active(RewardTermCfg))

    @property
    def _episode_sums(self) -> dict[str, torch.Tensor]:
        sums = self._env.buffers.logical("episode_sums")
        return {name: sums[:, k] for k, name in enumerate(self.active_terms)}

    @property
    def _step_reward(self) -> torch.Tensor:
        return self._env.buffers.logical("step_reward")

    def get_term_cfg(self, name: str) -> RewardTermCfg:
        return self._term_cfgs[name]

    def compute(self, dt: float | None = None) -> torch.Tensor:
        """Reward phase only (the fused ``env.step()`` normally covers it)."""
        env = self._env
        env.engine.step(env.buffers, phases=nat.PHASE_REWARDS, **env._rng_kwargs())
        return env.buffers.reward

    def evaluate_term(self, func, params: dict[str, Any]) -> torch.Tensor:
        """``func(env, **params)``: one reward term alone on the GPU (``rl_term_eval``)."""
        env = self._env
        term = compile_reward_term(func.__name__, RewardTermCfg(func=func, weight=1.0, params=params), env.spec.layout)
        return env.engine.term_eval(term, env.buffers, terminated=env.buffers.terminated)


class TerminationManager(_ManagerBase):
    def __init__(self, env):
        super().__init__(env)
        self.active_terms = [t.name for t in env.spec.dones]

    @property
    def terminated(self) -> torch.Tensor:
        return self._env.buffers.terminated.bool()

    @property
    def time_outs(self) -> torch.Tensor:
        return self._env.buffers.truncated.bool()

    @property
    def dones(self) -> torch.Tensor:
        return self.terminated | self.time_outs

    def get_term(self, name: str) -> torch.Tensor:
        return ((self._env.buffers.done_bits >> self.active_terms.index(name)) & 1).bool()

    def evaluate_term(self, func, params):
        raise NotImplementedError("termination terms are evaluated inside the fused step; read get_term(name)")


class CommandManager(_ManagerBase):
    def get_command(self, name: str) -> torch.Tensor:
        if name != "base_velocity":
            raise KeyError(name)
        return self._env.buffers.logical("command")

    def get_term(self, name: str):
        if name != "base_velocity":
            raise KeyError(name)
        return self._env.cfg.commands.base_velocity and _CommandTermView(self._env)

    def compute(self, dt: float | None = None) -> None:
        env = self._env
        env.engine.step(env.buffers, phases=nat.PHASE_COMMAND, **env._rng_kwargs())


class _CommandTermView:
    def __init__(self, env):
        self._env, self.cfg = env, env.cfg.commands.base_velocity

    @property
    def command(self):
        return self._env.buffers.logical("command")

    @property
    def metrics(self):
        b = self._env.buffers
        return {"error_vel_xy": b.logical("metric_error_vel_xy"), "error_vel_yaw": b.logical("metric_error_vel_yaw")}

    def __getattr__(self, name):
        if name in ("heading_target", "time_left", "is_heading_env", "is_standing_env"):
            return self._env.buffers.logical(name)
        raise AttributeError(name)


class ObservationManager(_ManagerBase):
    @property
    def group_obs_dim(self) -> dict[str, tuple[int, ...]]:
        return {g.name: (g.dim,) for g in self._env.spec.obs if g.dim > 0}

    def compute(self) -> dict[str, torch.Tensor]:
        env = self._env
        env.engine.step(env.buffers, phases=nat.PHASE_OBS, **env._rng_kwargs())
        return env._obs_dict()

    def evaluate_term(self, func, params):
        raise NotImplementedError("observation terms are evaluated inside the fused step; slice the group row instead")


_VELOCITY_KEYS = ("x", "y", "z", "roll", "pitch", "yaw")


def interval_push_terms(cfg) -> list[tuple[str, Any]]:
    """The active terms of ``cfg.events``, checked against what this env runs on the device: at most one non-global
    interval term calling ``push_by_setting_velocity`` [IL]. Anything else raises a ``ValueError`` naming the term -
    reset events write physical state through ``ResetEventStateProvider``, startup events belong to the simulator."""
    from .cfg import EventTermCfg
    from .mdp import push_by_setting_velocity

    events = getattr(cfg, "events", None)
    terms = [(n, t) for n, t in events.items() if t is not None] if events is not None else []
    for name, t in terms:
        if not isinstance(t, EventTermCfg):
            raise ValueError(f"event term '{name}': expected an EventTermCfg, got {type(t).__name__}")
        if t.mode != "interval":
            raise ValueError(f"event term '{name}': mode '{t.mode}' is not run by this env (reset events go through "
                             "ResetEventStateProvider, startup events belong to the simulator); only mode='interval'")
        if t.func is not push_by_setting_velocity:
            raise ValueError(f"event term '{name}': interval function {getattr(t.func, '__name__', t.func)!r} is not "
                             "supported; only push_by_setting_velocity")
        if t.is_global_time:
            raise ValueError(f"event term '{name}': is_global_time=True is not supported; only per-env interval timers")
        rng = t.interval_range_s
        if rng is None or len(rng) != 2 or not (float(rng[0]) <= float(rng[1])):
            raise ValueError(f"event term '{name}': interval_range_s must be (lo, hi) with lo <= hi, got {rng!r}")
        extra = set(t.params) - {"velocity_range", "asset_cfg"}
        if extra:
            raise ValueError(f"event term '{name}': unsupported params {sorted(extra)}")
        asset = t.params.get("asset_cfg")
        if asset is not None and getattr(asset, "name", None) != "robot":
            raise ValueError(f"event term '{name}': only the 'robot' asset can be pushed")
        vr = t.params.get("velocity_range", {})
        bad = set(vr) - set(_VELOCITY_KEYS)
        if bad:
            raise ValueError(f"event term '{name}': unknown velocity_range keys {sorted(bad)}; known: {list(_VELOCITY_KEYS)}")
        for k, (lo, hi) in vr.items():
            if not float(lo) <= float(hi):
                raise ValueError(f"event term '{name}': velocity_range['{k}'] needs lo <= hi, got {(lo, hi)!r}")
    if len(terms) > 1:
        raise ValueError(f"event terms {[n for n, _ in terms]}: one interval push term at most")
    return terms


class EventManager(_ManagerBase):
    """EventManager [IL] surface for the event terms this env runs: the interval push (stage 8 of ``env.step()``,
    ``rl_interval_push``). ``_interval_term_time_left`` holds one device timer tensor [N] per interval term, as
    upstream; the env owns the tensors."""

    def __init__(self, env, terms: list[tuple[str, Any]]):
        super().__init__(env)
        self._mode_term_names = {"interval": [n for n, _ in terms]} if terms else {}
        self._mode_term_cfgs = {"interval": [t for _, t in terms]} if terms else {}
        self._interval_term_time_left = [env.interval_time_left] if terms else []

    @property
    def available_modes(self) -> list[str]:
        return list(self._mode_term_names)

    @property
    def active_terms(self) -> dict[str, list[str]]:
        return dict(self._mode_term_names)

    def get_term_cfg(self, name: str):
        for names, cfgs in zip(self._mode_term_names.values(), self._mode_term_cfgs.values()):
            if name in names:
                return cfgs[names.index(name)]
        raise ValueError(f"event term '{name}' not found")


class _LazyLog(dict):
    """``extras["log"]``: a dict that fills itself from a snapshot of the device logging buffer on first access."""

    def __init__(self, env, snap: torch.Tensor):
        super().__init__()
        self._env, self._snap, self._built = env, snap, False

    def _fill(self):
        if not self._built:
            self._built = True
            super().update(self._env._build_log(self._snap))

    def __getitem__(self, k):
        self._fill()
        return super().__getitem__(k)

    def __contains__(self, k):
        self._fill()
        return super().__contains__(k)

    def __iter__(self):
        self._fill()
        return super().__iter__()

    def __len__(self):
        self._fill()
        return super().__len__()

    def keys(self):
        self._fill()
        return super().keys()

    def items(self):
        self._fill()
        return super().items()

    def values(self):
        self._fill()
        return super().values()

    def get(self, k, default=None):
        self._fill()
        return super().get(k, default)

    def __repr__(self):
        self._fill()
        return super().__repr__()


# --------------------------------------------------------------------------------------------------
# the env
# --------------------------------------------------------------------------------------------------
class ManagerBasedRLEnv:
    """Drop-in for ``isaaclab.envs.ManagerBasedRLEnv`` on the MDP side (no simulator attached)."""

    metadata = {"render_modes": [None]}

    def __init__(self, cfg, render_mode: str | None = None, state_provider: StateProvider | None = None,
                 body_tensors: str | None = None, rank: int = 0, **kwargs):
        self.cfg = cfg
        self.render_mode = render_mode
        self.device = torch.device(cfg.sim.device)
        self.num_envs = int(cfg.scene.num_envs)
        mode = body_tensors or cfg.scene.body_tensors
        layout = compact_layout(cfg) if mode == "compact" else cfg.scene.make_layout()
        self.spec = compile_step_spec(cfg, layout)
        self.engine = MdpStepEngine(self.spec, self.device)  # raises without the CUDA library: no CPU path
        self.buffers: StateBuffers = self.engine.new_buffers(self.num_envs)
        self.seed = int(getattr(cfg, "seed", 0) or 0)
        self.rank = rank
        self.step_dt = self.spec.step_dt
        self.physics_dt = cfg.sim.dt
        self.max_episode_length_s = cfg.episode_length_s
        self.max_episode_length = self.spec.max_episode_length
        self.common_step_counter = 0
        self.extras: dict[str, Any] = {}
        self._state_version = 0   # bumped whenever the physical state buffers change (derived views refresh lazily)
        self.scene = _Scene(self, terrain_origins=kwargs.get("terrain_origins"), terrain_types=kwargs.get("terrain_types"),
                            env_origins=kwargs.get("env_origins"))
        self.action_manager = ActionManager(self)
        self.observation_manager = ObservationManager(self)
        self.reward_manager = RewardManager(self)
        self.termination_manager = TerminationManager(self)
        self.command_manager = CommandManager(self)
        self.state_provider = state_provider or SyntheticStateProvider(self.spec, self.num_envs, self.device, seed=1234, rank=rank)
        self.single_observation_space = {g.name: Box(-math.inf, math.inf, (g.dim,)) for g in self.spec.obs if g.dim > 0}
        self.observation_space = {g.name: Box(-math.inf, math.inf, (self.num_envs, g.dim)) for g in self.spec.obs if g.dim > 0}
        self.single_action_space = Box(-math.inf, math.inf, (self.spec.A,))
        self.action_space = Box(-math.inf, math.inf, (self.num_envs, self.spec.A))
        # terrain-aware command restriction (V/mdp/commands.py:61-85): only when the terrain has a "pits" sub-terrain
        self.pit_grid = None
        from . import terrain as _terrain

        if _terrain.terrain_column_range(layout.terrain, "pits") is not None:
            self.pit_grid = _terrain.TerrainGridBuffers.create(layout.terrain, "pits", self.device,
                                                               origins=kwargs.get("terrain_origins"))
            self.was_on_pit = torch.zeros(self.num_envs, dtype=torch.uint8, device=self.device)
        self._all_ids = torch.arange(self.num_envs, dtype=torch.int32, device=self.device)
        self._n_all = torch.tensor([self.num_envs], dtype=torch.int32, device=self.device)
        # interval push (stage 8, randomize_push_robot): per-env timers sampled now, like EventManager._prepare_terms [IL]
        terms = interval_push_terms(cfg)
        self._push_cfg = MdpStepEngine.interval_event_cfg(terms[0][1]) if terms else None
        if terms:
            self.interval_time_left = torch.zeros(self.num_envs, dtype=torch.float32, device=self.device)
            self.pushed_ids = torch.zeros(self.num_envs, dtype=torch.int32, device=self.device)
            self.n_pushed = torch.zeros(1, dtype=torch.int32, device=self.device)
            self._reset_interval_timers()
        self.event_manager = EventManager(self, terms)
        self._closed = False

    # -- properties the scripts / wrapper read --------------------------------------------------------
    @property
    def unwrapped(self):
        return self

    @property
    def episode_length_buf(self) -> torch.Tensor:
        return self.buffers.t["episode_length"].long()

    @episode_length_buf.setter
    def episode_length_buf(self, value: torch.Tensor) -> None:
        self.buffers.t["episode_length"].copy_(value.to(self.device).to(torch.int32))

    @property
    def reset_buf(self) -> torch.Tensor:
        return self.termination_manager.dones

    @property
    def reward_buf(self) -> torch.Tensor:
        return self.buffers.reward

    def _rng_kwargs(self) -> dict:
        return dict(seed=self.seed, env_id_offset=self.rank * self.num_envs, use_random_inputs=False, use_step_counter=True)

    @property
    def _rng(self) -> dict:
        """``_rng_kwargs()`` cached (rebuilt when the seed changes): the hot loop does not build a dict per launch."""
        c = self.__dict__.get("_rng_cache")
        if c is None or c[0] != self.seed:
            c = (self.seed, self._rng_kwargs())
            self.__dict__["_rng_cache"] = c
        return c[1]

    def _obs_dict(self) -> dict[str, torch.Tensor]:
        return {g.name: self.buffers.obs[i] for i, g in enumerate(self.spec.obs) if g.dim > 0}

    def _log(self) -> "_LazyLog":
        """extras["log"] [IL]: the reset logging means of this step. The step wrote them into its own slot of the buffers'
        logging ring: no copy now, the ~30 named scalars only when somebody looks (rsl_rl reads them once per iteration,
        i.e. within the ring's 64 steps)."""
        return _LazyLog(self, self.buffers.log_all)

    def _build_log(self, snap: torch.Tensor) -> dict[str, torch.Tensor]:
        log, kk = {}, max(self.spec.K, 1)
        sums = snap[:kk] / self.max_episode_length_s
        for k, name in enumerate(self.reward_manager.active_terms):
            log[f"Episode_Reward/{name}"] = sums[k]
        for i, name in enumerate(self.termination_manager.active_terms):
            log[f"Episode_Termination/{name}"] = snap[kk + i]
        log["Metrics/base_velocity/error_vel_xy"] = snap[kk + nat.RL_MAX_DONE_TERMS]
        log["Metrics/base_velocity/error_vel_yaw"] = snap[kk + nat.RL_MAX_DONE_TERMS + 1]
        return log

    def _push_rng(self) -> dict:
        return dict(seed=self.seed, env_id_offset=self.rank * self.num_envs, use_step_counter=True)

    def _reset_interval_timers(self) -> None:
        """EventManager.reset(all ids) [IL]: fresh interval timers for every env."""
        self.engine.interval_push(self.buffers, self._push_cfg, self.interval_time_left, env_ids=self._all_ids,
                                  n_env_ids=self._n_all, **self._push_rng())

    def _interval_push(self) -> None:
        """Stage 8, event_manager.apply("interval") [IL]: after the command update, before the observations. The
        pushed envs are ``pushed_ids[:n_pushed]`` - a simulator writes their root velocities into the simulation."""
        self.engine.interval_push(self.buffers, self._push_cfg, self.interval_time_left, pushed_ids=self.pushed_ids,
                                  n_pushed=self.n_pushed, **self._push_rng())

    def invalidate_derived(self) -> None:
        """Call after writing physical state into ``buffers`` by hand: the derived articulation views refresh lazily."""
        self._state_version += 1

    # -- gym API -------------------------------------------------------------------------------------------
    def reset(self, seed: int | None = None, options: dict | None = None):
        """Reset every env: provider state, manager reset of all ids, command compute, observations."""
        if seed is not None:
            self.seed = int(seed)
        b = self.buffers
        self.state_provider.advance(self)
        self.state_provider.reset(self, self._all_ids, self._n_all)
        if self._push_cfg is not None:
            self._reset_interval_timers()
        self._state_version += 1
        b.done_bits.zero_()
        self.engine.step(b, phases=nat.PHASE_RESET | nat.PHASE_COMMAND | nat.PHASE_OBS, env_ids=self._all_ids,
                         n_env_ids=self._n_all, **self._rng_kwargs())
        self.extras = {"log": self._log()}
        return self._obs_dict(), self.extras

    def step(self, action: torch.Tensor):
        """ManagerBasedRLEnv.step() [IL] order (SURVEY.md 3.2): three launches of this library + the provider."""
        b, eng = self.buffers, self.engine
        eng.pin_stream()   # one stream lookup for the three launches of the step
        try:
            nvtx = _NVTX   # RL_MDP_NVTX=1: ranges around the launches for nsys / ncu timelines (SURVEY.md section 5, "Tracing")
            if nvtx:
                torch.cuda.nvtx.range_push("mdp.process_action")
            self.action_manager.process_action(action)                                   # 1 (+ common step counter)
            if nvtx:
                torch.cuda.nvtx.range_pop()
                torch.cuda.nvtx.range_push("mdp.state_provider.advance")
            self.state_provider.advance(self)                                            # 2 physics / sensors
            self.common_step_counter += 1
            if nvtx:
                torch.cuda.nvtx.range_pop()
                torch.cuda.nvtx.range_push("mdp.step_pre_reset")
            eng.step_pre_reset(b, **self._rng)                                           # 3-5: dones, rewards, reset ids
            if nvtx:
                torch.cuda.nvtx.range_pop()
            self.state_provider.reset(self, b.reset_ids, b.n_reset)                      # 6a external reset
            self._state_version += 1
            b.advance_log_slot()
            if nvtx:
                torch.cuda.nvtx.range_push("mdp.step_post_reset")
            push = self._push_cfg is not None
            if self.pit_grid is None:
                eng.step_post_reset(b, **self._rng)                                      # 6b manager reset, 7 command, 9 obs
                if push:   # 8 after the fused launch: the pushed envs' observation rows are written again
                    self._interval_push()
                    eng.reobserve(b, self.pushed_ids, self.n_pushed, **self._rng)
            else:   # the pit branch of _update_command sits between the command update and the observations
                rng = self._rng
                eng.step(b, phases=nat.PHASE_RESET | nat.PHASE_COMMAND, **rng)
                eng.command_pit_restrict(b, self.pit_grid, self.was_on_pit, **rng)
                if push:
                    self._interval_push()                                                # 8
                eng.step(b, phases=nat.PHASE_OBS, **rng)
            if push:
                self._state_version += 1
            if nvtx:
                torch.cuda.nvtx.range_pop()
        finally:
            eng.unpin_stream()
        self.extras = {"log": self._log()}
        return self._obs_dict(), b.reward, b.terminated.view(torch.bool), b.truncated.view(torch.bool), self.extras   # 0/1 bytes: views, no kernels

    def close(self) -> None:
        if not self._closed:
            self.engine.close()
            self._closed = True

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class RslRlVecEnvWrapper:
    """``isaaclab_rl.rsl_rl.RslRlVecEnvWrapper`` [IL] surface: what rsl_rl's OnPolicyRunner calls."""

    def __init__(self, env: ManagerBasedRLEnv, clip_actions: float | None = None):
        if not isinstance(env.unwrapped, ManagerBasedRLEnv):
            raise ValueError(f"The environment must be inherited from ManagerBasedRLEnv. Environment type: {type(env)}")
        self.env = env
        self.clip_actions = clip_actions
        self.num_envs = env.unwrapped.num_envs
        self.device = env.unwrapped.device
        self.max_episode_length = env.unwrapped.max_episode_length
        self.num_actions = env.unwrapped.action_manager.total_action_dim
        self._dones = None
        self.env.reset()

    def __str__(self):
        return f"<{type(self).__name__}{self.env}>"

    @classmethod
    def class_name(cls) -> str:
        return cls.__name__

    @property
    def cfg(self):
        return self.unwrapped.cfg

    @property
    def unwrapped(self) -> ManagerBasedRLEnv:
        return self.env.unwrapped

    @property
    def observation_space(self):
        return self.env.observation_space

    @property
    def action_space(self):
        return self.env.action_space

    @property
    def episode_length_buf(self) -> torch.Tensor:
        return self.unwrapped.episode_length_buf

    @episode_length_buf.setter
    def episode_length_buf(self, value: torch.Tensor):
        self.unwrapped.episode_length_buf = value

    def seed(self, seed: int = -1) -> int:
        self.unwrapped.seed = seed
        return seed

    def _pack(self, obs: dict[str, torch.Tensor]):
        if TensorDict is not None:
            return TensorDict(obs, batch_size=[self.num_envs])
        return obs

    def reset(self):
        obs, extras = self.env.reset()
        return self._pack(obs), extras

    def get_observations(self):
        return self._pack(self.unwrapped._obs_dict())

    def step(self, actions: torch.Tensor):
        if self.clip_actions is not None:
            actions = torch.clamp(actions, -self.clip_actions, self.clip_actions)
        obs, rew, terminated, truncated, extras = self.env.step(actions)
        if self._dones is None or self._dones.shape != terminated.shape:
            self._dones = torch.empty(terminated.shape, dtype=torch.long, device=terminated.device)
        b = self.unwrapped.buffers
        dones = torch.bitwise_or(b.terminated, b.truncated, out=self._dones)   # uint8 | uint8 -> long, one kernel
        if not getattr(self.unwrapped.cfg, "is_finite_horizon", False):
            extras["time_outs"] = truncated
        return self._pack(obs), rew, dones, extras

    def close(self):
        return self.env.close()


def make(task: str, cfg=None, num_envs: int | None = None, device: str | None = None, **kwargs) -> ManagerBasedRLEnv:
    """``gym.make(task, cfg=env_cfg)`` equivalent (V/config/quadruped/unitree_go2/__init__.py:12-32)."""
    from .tasks import make_env_cfg

    if cfg is None:
        cfg = make_env_cfg(task, num_envs)
    elif num_envs is not None:
        cfg.scene.num_envs = int(num_envs)
    if device is not None:
        cfg.sim.device = device
    return ManagerBasedRLEnv(cfg, **kwargs)


if gym is not None:  # pragma: no cover - registration under the reference's ids when gymnasium exists
    from .tasks import TASKS as _TASKS

    for _task in _TASKS:
        try:
            gym.register(id=_task, entry_point="robot_lab_b200.envs:ManagerBasedRLEnv", disable_env_checker=True,
                         kwargs={"env_cfg_entry_point": f"robot_lab_b200.tasks:TASKS['{_task}']"})
        except Exception:
            pass
