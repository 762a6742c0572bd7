"""SURVEY.md 8(b).2: the env surface term functions read. Two UNMODIFIED reference term functions (loaded from
/root/reference through oracle/isaaclab_shim.py) run against THIS repo's scene classes (robot_lab_b200.envs._Scene and
friends: field names, aliases, shapes, SceneEntityCfg resolution, sensors dict, terrain object) and must reproduce the
oracle's term values. Build container only: the device side of the same surface - the CUDA-computed derived views and
rl_term_eval - is tests/test_gpu_env_surface.py, which needs no reference files."""

import types

import pytest
import torch

import helpers as H
from oracle import isaaclab_shim, mdp_port as port
from robot_lab_b200.synthetic import make_state

needs_reference = pytest.mark.skipif(not isaaclab_shim.reference_available(), reason="needs the robot_lab source tree")


class _CpuBuffers:
    """StateBuffers.logical() over the logical CPU tensors of the synthetic state (no device, no kernels)."""

    def __init__(self, spec, st):
        self.spec, self.st, self.N = spec, st, st["root_quat_w"].shape[0]

    def logical(self, name):
        x = self.st[name]
        if name == "net_forces_w_history":
            return x.reshape(self.N, self.spec.T, self.spec.B, 3)
        if name in ("body_pos_w", "body_lin_vel_w"):
            return x.reshape(self.N, self.spec.Ba, 3)
        return x


def _cpu_env(cfg, spec, st):
    """The attributes robot_lab_b200.envs' scene classes need from an env, on the CPU: derived articulation views come
    from the oracle here (on a GPU they are filled by rl_derived_views)."""
    from robot_lab_b200 import envs

    n = st["root_quat_w"].shape[0]
    env = types.SimpleNamespace(num_envs=n, device=torch.device("cpu"), spec=spec, cfg=cfg, buffers=_CpuBuffers(spec, st),
                                step_dt=spec.step_dt, state_provider=None, _state_version=0)
    d = port.Derived(st, spec)

    def refresh(self):
        self._vec[0], self._vec[1], self._vec[2] = d.projected_gravity_b, d.root_lin_vel_b, d.root_ang_vel_b
        self._heading.copy_(d.heading_w())

    orig = envs._ArticulationData._refresh
    envs._ArticulationData._refresh = refresh
    try:
        env.scene = envs._Scene(env)
    finally:
        pass
    env._restore = lambda: setattr(envs._ArticulationData, "_refresh", orig)
    env.command_manager = types.SimpleNamespace(get_command=lambda name: st["command"])
    env.action_manager = types.SimpleNamespace(action=st["action"], prev_action=st["prev_action"])
    env.episode_length_buf = st["episode_length"].long()
    return env


def _full_spec(key):
    return H.make_spec(key, full_layout=True)   # every tensor carries every body, IsaacLab-style


@pytest.fixture
def go2_env():
    cfg, spec = _full_spec("go2_rough")
    st = make_state(spec, 300, seed=21)
    env = _cpu_env(cfg, spec, st)
    yield cfg, spec, st, env
    env._restore()


@needs_reference
def test_unmodified_track_lin_vel_xy_exp_runs_on_this_scene(go2_env):
    """V/mdp/rewards.py:22-35 reads env.scene[name].data.{root_lin_vel_b, projected_gravity_b} and the command manager."""
    from robot_lab_b200.cfg import SceneEntityCfg

    cfg, spec, st, env = go2_env
    ref = isaaclab_shim.load_reference_module("rewards.py")
    asset_cfg = SceneEntityCfg("robot")
    asset_cfg.resolve(env.scene)
    got = ref.track_lin_vel_xy_exp(env, std=0.5, command_name="base_velocity", asset_cfg=asset_cfg)
    t = next(t for t in spec.rewards if t.type_name == "track_lin_vel_xy_exp")
    torch.testing.assert_close(got, port.reward_term(t, st, spec), rtol=1e-6, atol=1e-6)


@needs_reference
def test_unmodified_feet_slide_runs_on_this_scene(go2_env):
    """V/mdp/rewards.py:557-587 reads env.scene.sensors[name].data.net_forces_w_history[:, :, body_ids], the asset's
    body_lin_vel_w[:, body_ids], root_lin_vel_w, root_quat_w and projected_gravity_b; the ids come from
    SceneEntityCfg(body_names=...).resolve(scene)."""
    from robot_lab_b200.cfg import SceneEntityCfg

    cfg, spec, st, env = go2_env
    ref = isaaclab_shim.load_reference_module("rewards.py")
    sensor_cfg = SceneEntityCfg("contact_forces", body_names=".*_foot")
    asset_cfg = SceneEntityCfg("robot", body_names=".*_foot")
    sensor_cfg.resolve(env.scene)
    asset_cfg.resolve(env.scene)
    assert len(sensor_cfg.body_ids) == 4 and len(asset_cfg.body_ids) == 4
    got = ref.feet_slide(env, sensor_cfg=sensor_cfg, asset_cfg=asset_cfg)
    t = next(t for t in spec.rewards if t.type_name == "feet_slide")
    torch.testing.assert_close(got, port.reward_term(t, st, spec), rtol=1e-5, atol=1e-6)


@needs_reference
def test_unmodified_terrain_utils_read_this_scene_terrain(go2_env):
    """V/mdp/utils.py:44-127 reads env.scene.terrain.{cfg.terrain_type, cfg.terrain_generator, terrain_types,
    terrain_origins}: the in-scope terrains have no "pits" sub-terrain -> both helpers return all-False."""
    cfg, spec, st, env = go2_env
    utils = isaaclab_shim.load_reference_module("utils.py")
    assert env.scene.terrain.cfg.terrain_type == "generator"
    assert tuple(env.scene.terrain.terrain_origins.shape) == (10, 20, 3)
    assert tuple(env.scene.env_origins.shape) == (300, 3)
    assert not utils.is_env_assigned_to_terrain(env, "pits").any()
    assert not utils.is_robot_on_terrain(env, "pits").any()
    # a sub-terrain that exists: the assignment follows terrain_types, the position test the grid of origins
    mask = utils.is_env_assigned_to_terrain(env, "boxes")
    col = env.scene.terrain.terrain_types
    assert torch.equal(mask, (col >= 8) & (col < 12))


def test_height_scanner_surface(go2_env):
    """The height_scan observation [IL] = sensor.data.pos_w[:, 2:3] - sensor.data.ray_hits_w[..., 2] - offset."""
    cfg, spec, st, env = go2_env
    sensor = env.scene.sensors["height_scanner"]
    assert tuple(sensor.data.pos_w.shape) == (300, 3) and tuple(sensor.data.ray_hits_w.shape) == (300, spec.R, 3)
    hs = sensor.data.pos_w[:, 2].unsqueeze(1) - sensor.data.ray_hits_w[..., 2] - 0.5
    torch.testing.assert_close(hs, st["ray_sensor_pos_z"].reshape(-1, 1) - st["ray_hits_z"] - 0.5, rtol=0, atol=0)
    # the hit points sit on the yaw-aligned 17 x 11 grid around the sensor
    d = (sensor.data.ray_hits_w[..., :2] - sensor.data.pos_w[:, None, :2]).norm(dim=-1)
    assert d.max() <= (0.8 ** 2 + 0.5 ** 2) ** 0.5 + 1e-4
