"""CPU checks of the oracle restatements for SURVEY.md 8(f) rows 3 and 4 (actuator models, terrain-aware command
restriction, pit branch of the reset event, height-scan casting).

robot_lab-owned pieces (V/mdp/utils.py, V/mdp/commands.py:49-85, V/mdp/events.py:232-244) are pinned against the stored
outputs of the unmodified reference files (tests/golden/pit_terrain_*.npz, reference_pins.npz); the IsaacLab-owned
ones (actuator models, ray caster) are PARITY UNPINNED and checked against hand-computed / analytic values."""

import math
from pathlib import Path

import numpy as np
import pytest
import torch

import helpers as H
from oracle import mdp_port as port
from robot_lab_b200 import terrain as terrain_host
from robot_lab_b200.assets import ASSETS
from robot_lab_b200.cfg import RayCasterCfg, ResetStateCfg, TerrainCfg
from robot_lab_b200.synthetic import make_state

CMD_KEYS = ("command", "heading_target", "time_left", "is_heading_env", "is_standing_env", "metric_error_vel_xy",
            "metric_error_vel_yaw")
PIT_TERRAIN = TerrainCfg(sub_terrains=("pyramid_stairs", "pits", "boxes", "random_rough", "hf_pyramid_slope"),
                         proportions=(0.2, 0.15, 0.25, 0.3, 0.1))


# ---- actuator models [IL] --------------------------------------------------------------------------------------
def test_dc_motor_hand_checked_go2():
    """Go2 'legs' DCMotor (assets/unitree.py:107-115): kp 25, kd 0.5, effort 23.5 = saturation, no-load speed 30."""
    tab = ASSETS["unitree_go2"].actuator_table()
    assert set(tab["kind"]) == {"dc_motor"} and tab["stiffness"][0] == 25.0 and tab["velocity_limit"][0] == 30.0
    J = 12
    q = torch.zeros(5, J)
    tgt = torch.tensor([0.1, 1.0, 1.0, -1.0, 2.0]).unsqueeze(1).repeat(1, J)
    qd = torch.tensor([0.0, 30.0, -30.0, 15.0, 0.0]).unsqueeze(1).repeat(1, J)
    computed, applied = port.actuator_step(tab, tgt, q, qd)
    # row 0: small error, inside every limit
    assert torch.allclose(computed[0], torch.full((J,), 2.5)) and torch.equal(applied[0], computed[0])
    # row 1: at +no-load speed the motor cannot push forward: max effort = sat * (1 - 1) = 0
    assert torch.allclose(computed[1], torch.full((J,), 25.0 - 15.0)) and torch.equal(applied[1], torch.zeros(J))
    # row 2: at -no-load speed the forward limit is the effort limit (top = 2 * sat, clipped to 23.5)
    assert torch.allclose(computed[2], torch.full((J,), 25.0 + 15.0)) and torch.allclose(applied[2], torch.full((J,), 23.5))
    # row 3: braking torque at half speed: bottom = sat * (-1 - 0.5) = -35.25 -> min effort -23.5; computed -32.5
    assert torch.allclose(applied[3], torch.full((J,), -23.5))
    # row 4: standing still, large error: plain effort limit
    assert torch.allclose(applied[4], torch.full((J,), 23.5))


def test_implicit_actuator_g1_table():
    a = ASSETS["unitree_g1_29dof"]
    tab = a.actuator_table()
    assert set(tab["kind"]) == {"implicit"}
    j = a.joint_names.index("left_knee_joint")
    # assets/unitree.py:456-464, 508-536: STIFFNESS_7520_22 / DAMPING_7520_22, effort 139
    w = 10 * 2.0 * 3.1415926535
    assert math.isclose(tab["stiffness"][j], 0.025101925 * w**2, rel_tol=1e-12)
    assert math.isclose(tab["damping"][j], 2.0 * 2.0 * 0.025101925 * w, rel_tol=1e-12)
    assert tab["effort_limit"][j] == 139.0
    q, qd = torch.zeros(2, 29), torch.zeros(2, 29)
    tgt = torch.zeros(2, 29)
    tgt[0, j], tgt[1, j] = 0.5, 3.0
    computed, applied = port.actuator_step(tab, tgt, q, qd)
    assert torch.allclose(computed[0, j], torch.tensor(0.5 * tab["stiffness"][j])) and applied[0, j] == computed[0, j]
    assert applied[1, j] == 139.0 and computed[1, j] > 139.0


# ---- terrain queries (V/mdp/utils.py) -----------------------------------------------------------------------------
def test_terrain_column_range_host_and_oracle_agree():
    for ter in (PIT_TERRAIN, TerrainCfg()):
        for name in ("pits", "boxes", "pyramid_stairs", "hf_pyramid_slope"):
            assert terrain_host.terrain_column_range(ter, name) == port.terrain_column_range(
                list(ter.sub_terrains), list(ter.proportions), ter.num_cols, name)
    assert terrain_host.terrain_column_range(PIT_TERRAIN, "pits") == (4, 7)
    assert terrain_host.terrain_column_range(TerrainCfg(), "pits") is None
    assert terrain_host.terrain_column_range(TerrainCfg(terrain_type="plane"), "boxes") is None


def _pit_golden(key):
    """Seeded inputs on PIT_TERRAIN and the outputs of the reference's own functions for them (make_golden.py::pits)."""
    z = np.load(Path(__file__).resolve().parent / "golden" / f"pit_terrain_{key}.npz")
    return {k: torch.from_numpy(z[k]) for k in z.files}


def test_terrain_utils_match_reference_functions():
    """_get_terrain_column_range / is_env_assigned_to_terrain of the unmodified V/mdp/utils.py for a sub-terrain at the
    start, in the middle and at the end of the list and for a missing one (reference_pins.npz), is_robot_on_terrain
    on the pit-terrain fixtures."""
    pins = H.reference_pins()
    pos, types, origins = H.terrain_query_inputs(PIT_TERRAIN)
    for name in ("pits", "boxes", "random_rough", "nope"):
        rng = terrain_host.terrain_column_range(PIT_TERRAIN, name)
        assert (rng if rng is not None else (-1, -1)) == tuple(pins[f"terrain/{name}/column_range"].tolist()), name
        assert torch.equal(terrain_host.is_env_assigned_to_terrain(PIT_TERRAIN, types, name).bool(),
                           pins[f"terrain/{name}/assigned"]), name
    assert port.is_robot_on_terrain(pos, origins, (4, 7)).float().mean() > 0.05
    for key in ("go2_rough", "g1_rough"):
        z = _pit_golden(key)
        for name in ("pits", "boxes"):
            rng = terrain_host.terrain_column_range(PIT_TERRAIN, name)
            got = port.is_robot_on_terrain(z["in/root_pos_w"], z["terrain_origins"], rng)
            assert torch.equal(got, z[f"on_terrain/{name}"]), (key, name)


@pytest.mark.parametrize("key", ["go2_rough", "g1_rough"])
def test_pit_command_branch_matches_reference_class(key):
    """Two consecutive CommandTerm.compute() calls of the unmodified UniformThresholdVelocityCommand on a terrain with
    a "pits" sub-terrain; the robots move between the calls, so that some enter, stay on and leave the pits (reference
    output of both calls in reference_pins.npz)."""
    cfg, spec = H.make_spec(key)
    pins = H.reference_pins()
    n = 2048
    st = make_state(spec, n, seed=21)
    g = torch.Generator().manual_seed(4)
    origins = terrain_host.grid_origins(PIT_TERRAIN)
    rng = terrain_host.terrain_column_range(PIT_TERRAIN, "pits")
    was = torch.rand(n, generator=g) < 0.3
    u = st["cmd_uniforms"]
    n_left = n_on = 0
    for it in range(2):
        st["root_pos_w"] = H.pit_positions(n, g)
        got = port.compute_command(spec, st, {"cmd_uniforms": u})
        on = port.is_robot_on_terrain(st["root_pos_w"], origins, rng)
        assert torch.equal(on, pins[f"pit_steps/{key}/{it}/was_on_pit"])
        n_left += int((was & ~on).sum())
        n_on += int(on.sum())
        got.update(port.command_pit_restrict(spec, {**st, **got}, on, was, u))
        for k in CMD_KEYS + ("was_on_pit",):
            assert torch.equal(got[k], pins[f"pit_steps/{key}/{it}/{k}"]), (it, k)
        st.update({k: got[k] for k in CMD_KEYS})
        was = got["was_on_pit"]
    assert n_left > 50 and n_on > 100


def test_reset_root_state_pit_branch_matches_reference():
    cfg, spec = H.make_spec("go2_rough")
    z = _pit_golden("go2_rough")
    st = {k[3:]: v for k, v in z.items() if k.startswith("in/")}
    n = st["root_pos_w"].shape[0]
    st.update(joint_pos=torch.zeros(n, spec.J), joint_vel=torch.zeros(n, spec.J))
    pits = terrain_host.is_env_assigned_to_terrain(PIT_TERRAIN, z["terrain_types"], "pits")
    ids = z["reset/ids"]
    assert 0 < int(pits[ids.long()].sum()) < len(ids)
    got = port.reset_scene_state(spec, st, ids, ResetStateCfg.go2_rough(), z["reset/env_origins"], z["reset/uniforms"],
                                 assigned_to_pits=pits)
    for k in ("root_pos_w", "root_quat_w", "root_lin_vel_w", "root_ang_vel_w"):
        torch.testing.assert_close(got[k][ids.long()], z[f"reset/out/{k}"], rtol=0, atol=0, msg=k)


# ---- height scanner [IL] -----------------------------------------------------------------------------------------
def test_grid_pattern_matches_cfg():
    rc = RayCasterCfg()
    s = terrain_host.grid_pattern_ray_starts(rc)
    assert s.shape == (187, 3) and rc.num_rays == 187
    assert torch.equal(s, port.grid_pattern_ray_starts(rc.size, rc.resolution, rc.offset_z))
    # x fastest: first 17 rays share y = -0.5
    assert torch.all(s[:17, 1] == s[0, 1]) and abs(float(s[0, 0]) + 0.8) < 1e-6 and abs(float(s[16, 0]) - 0.8) < 1e-6
    assert abs(float(s[-1, 1]) - 0.5) < 1e-6 and torch.all(s[:, 2] == 20.0)


def test_height_scan_on_a_plane_and_outside():
    """A planar height field is reproduced exactly (up to fp32 rounding) by both triangles; rays that leave the field
    return +inf."""
    nx, ny, hs = 96, 80, 0.1
    a, b, c = 0.3, -0.2, 1.5
    xs, ys = torch.arange(nx) * hs - 3.0, torch.arange(ny) * hs - 3.0
    heights = a * xs[:, None] + b * ys[None, :] + c
    starts = terrain_host.grid_pattern_ray_starts(RayCasterCfg())
    g = torch.Generator().manual_seed(0)
    n = 64
    pos = torch.stack([torch.rand(n, generator=g) * 2.0 - 0.5, torch.rand(n, generator=g) * 1.5 - 0.2,
                       torch.rand(n, generator=g)], dim=1)
    pos[0, :2] = torch.tensor([-3.4, 0.0])      # partially outside
    pos[1, :2] = torch.tensor([40.0, 40.0])     # completely outside
    quat = torch.nn.functional.normalize(torch.randn(n, 4, generator=g), dim=1)
    z, sz = port.height_scan_cast(heights, -3.0, -3.0, hs, starts, pos, quat)
    assert z.shape == (n, 187) and torch.equal(sz, pos[:, 2])
    assert torch.isinf(z[1]).all() and torch.isinf(z[0]).any() and torch.isfinite(z[2:]).all()
    # world xy of the rays from the yaw-only rotation
    yaw = torch.atan2(2 * (quat[:, 0] * quat[:, 3] + quat[:, 1] * quat[:, 2]), 1 - 2 * (quat[:, 2] ** 2 + quat[:, 3] ** 2))
    wx = pos[:, 0:1] + torch.cos(yaw)[:, None] * starts[None, :, 0] - torch.sin(yaw)[:, None] * starts[None, :, 1]
    wy = pos[:, 1:2] + torch.sin(yaw)[:, None] * starts[None, :, 0] + torch.cos(yaw)[:, None] * starts[None, :, 1]
    want = a * wx + b * wy + c
    torch.testing.assert_close(z[2:], want[2:], rtol=0, atol=2e-5)
