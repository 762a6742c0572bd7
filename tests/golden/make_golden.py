"""Generate the committed golden fixtures by running the REFERENCE's own functions (unmodified files under
/root/reference, loaded through oracle/isaaclab_shim.py) on seeded synthetic state.

    python tests/golden/make_golden.py          # build container only (needs /root/reference)

Each ``<task>.npz`` holds: the synthetic input state (logical shapes, fp32), the raw value of every reward term
the reference owns (V/mdp/rewards.py functions incl. the GaitReward class), the reference's
UniformThresholdVelocityCommand.compute() result (V/mdp/commands.py over a restated [IL] base class) and the two
reference observation functions (V/mdp/observations.py). IsaacLab-owned terms have no reference source
("parity unpinned", oracle/mdp_port.py) and are NOT in the fixtures.
"""
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

import helpers as H  # noqa: E402
from oracle import isaaclab_shim, ref_harness  # noqa: E402
from robot_lab_b200.synthetic import make_state  # noqa: E402

N = {"a1_flat": 64, "go2_flat": 48, "go2_rough": 48, "g1_rough": 48, "g1_rough_37": 32}
SEED = 20260922


def main():
    assert isaaclab_shim.reference_available(), "needs /root/reference"
    out_dir = Path(__file__).resolve().parent
    for key, n in list(N.items()) + [("go2_catalogue", 48)]:
        cfg, spec = H.make_catalogue_spec() if key == "go2_catalogue" else H.make_spec(key)
        st = make_state(spec, n, seed=SEED)
        arrays = {f"in/{k}": v.numpy() for k, v in st.items()}
        for name, val in ref_harness.reference_reward_terms(cfg, spec, st).items():
            if val is not None:
                arrays[f"reward/{name}"] = val.float().numpy()
        ter = "plane" if "flat" in key else "generator"
        if key == "go2_catalogue":
            np.savez_compressed(out_dir / f"{key}.npz", **arrays)
            print(key, n, "envs,", sum(1 for k in arrays if k.startswith("reward/")), "reference-owned reward terms")
            continue
        for name, val in ref_harness.reference_command_compute(spec, st, st["cmd_uniforms"], ter).items():
            if name != "was_on_pit":   # all False without a "pits" sub-terrain; pit_terrain_*.npz covers that branch
                arrays[f"command/{name}"] = val.numpy()
        obs = ref_harness.reference_observation_terms(spec, st)
        arrays["obs/phase"] = obs["phase"].numpy()
        arrays["obs/joint_pos_rel_without_wheel"] = obs["joint_pos_rel_without_wheel"].numpy()
        arrays["obs/_wheel_ids"] = obs["_wheel_ids"].numpy()
        np.savez_compressed(out_dir / f"{key}.npz", **arrays)
        print(key, n, "envs,", sum(1 for k in arrays if k.startswith("reward/")), "reference-owned reward terms")


def reset_event():
    """reset_state_<task>.npz: inputs (ids, uniforms, env origins) and what the reference's reset_root_state_uniform
    (V/mdp/events.py:205-271) writes into the simulator for them (Go2 rough ranges, GO2/rough_env_cfg.py:56-73)."""
    from robot_lab_b200.cfg import ResetStateCfg

    out_dir = Path(__file__).resolve().parent
    for key, n in (("go2_rough", 96), ("g1_rough", 40)):
        cfg, spec = H.make_spec(key)
        st = make_state(spec, n, seed=SEED)
        g = torch.Generator().manual_seed(SEED + 1)
        uniforms = torch.rand(12 + 2 * spec.J, n, generator=g)
        origins = torch.randn(n, 3, generator=g) * 20.0
        ids = torch.randperm(n, generator=g)[: n // 3].sort().values.int()
        ref = ref_harness.reference_reset_root_state(spec, st, ids, ResetStateCfg.go2_rough(), origins, uniforms)
        arrays = {"ids": ids.numpy(), "uniforms": uniforms.numpy(), "env_origins": origins.numpy()}
        arrays.update({f"out/{k}": v.numpy() for k, v in ref.items()})
        np.savez_compressed(out_dir / f"reset_state_{key}.npz", **arrays)
        print("reset_state", key, n, "envs,", len(ids), "reset")


PIT_SUB_TERRAINS = ("pyramid_stairs", "pits", "boxes", "random_rough", "hf_pyramid_slope")
PIT_PROPORTIONS = (0.2, 0.15, 0.25, 0.3, 0.1)


def pits():
    """pit_terrain_<task>.npz: a generator terrain WITH a "pits" sub-terrain (none of the reference's task configs
    has one, so the golden vectors of main() never reach that code): the reference's is_robot_on_terrain /
    is_env_assigned_to_terrain (V/mdp/utils.py:44-127), UniformThresholdVelocityCommand.compute() with the pit
    branch of _update_command live (V/mdp/commands.py:61-85) and the pit branch of reset_root_state_uniform
    (V/mdp/events.py:232-244)."""
    from robot_lab_b200 import terrain as terrain_host
    from robot_lab_b200.cfg import ResetStateCfg, TerrainCfg

    out_dir = Path(__file__).resolve().parent
    ter_cfg = TerrainCfg(sub_terrains=PIT_SUB_TERRAINS, proportions=PIT_PROPORTIONS)
    for key, n in (("go2_rough", 512), ("g1_rough", 256)):
        cfg, spec = H.make_spec(key)
        st = make_state(spec, n, seed=SEED + 7)
        g = torch.Generator().manual_seed(SEED + 8)
        st["root_pos_w"] = torch.stack([(torch.rand(n, generator=g) - 0.5) * 70.0, (torch.rand(n, generator=g) - 0.5) * 150.0,
                                        torch.rand(n, generator=g)], dim=1)
        origins = terrain_host.grid_origins(ter_cfg)
        origins[:, :, 2] = torch.rand(origins.shape[:2], generator=g)
        types = torch.randint(0, ter_cfg.num_cols, (n,), generator=g)
        was = torch.rand(n, generator=g) < 0.35
        ter = ref_harness.fake_terrain(ter_cfg, "generator", n, origins, types)
        keep = ("root_pos_w", "root_quat_w", "root_lin_vel_w", "root_ang_vel_w", "command", "heading_target", "time_left",
                "is_heading_env", "is_standing_env", "metric_error_vel_xy", "metric_error_vel_yaw", "cmd_uniforms")
        arrays = {f"in/{k}": st[k].numpy() for k in keep}   # everything the command term and the reset event read
        arrays.update({"terrain_origins": origins.numpy(), "terrain_types": types.numpy(), "was_on_pit": was.numpy()})
        ref = ref_harness.reference_command_compute(spec, st, st["cmd_uniforms"], "generator", terrain=ter, was_on_pit=was)
        arrays.update({f"command/{k}": v.numpy() for k, v in ref.items()})
        utils = ref_harness.reference_terrain_utils()
        env = ref_harness.FakeEnv(spec, st)
        env.scene.terrain = ter
        for name in ("pits", "boxes"):
            arrays[f"on_terrain/{name}"] = utils.is_robot_on_terrain(env, name).numpy()
            arrays[f"assigned/{name}"] = utils.is_env_assigned_to_terrain(env, name).numpy()
        uniforms = torch.rand(12 + 2 * spec.J, n, generator=g)
        env_origins = torch.randn(n, 3, generator=g) * 20.0
        ids = torch.randperm(n, generator=g)[: n // 3].sort().values.int()
        rr = ref_harness.reference_reset_root_state(spec, st, ids, ResetStateCfg.go2_rough(), env_origins, uniforms, terrain=ter)
        arrays.update({"reset/ids": ids.numpy(), "reset/uniforms": uniforms.numpy(), "reset/env_origins": env_origins.numpy()})
        arrays.update({f"reset/out/{k}": v.numpy() for k, v in rr.items()})
        np.savez_compressed(out_dir / f"pit_terrain_{key}.npz", **arrays)
        print("pit_terrain", key, n, "envs,", int(ref["was_on_pit"].sum()), "on pits,", int((was & ~ref["was_on_pit"]).sum()), "left a pit")


EDGE_KEYS = ("go2_rough", "a1_flat")
RESET_KEYS = ("go2_rough", "g1_rough")
PIT_STEP_KEYS = ("go2_rough", "g1_rough")
RANGE_NAMES = ("pits", "boxes", "random_rough", "nope")
CMD_KEYS = ("command", "heading_target", "time_left", "is_heading_env", "is_standing_env", "metric_error_vel_xy",
            "metric_error_vel_yaw")
ROOT_KEYS = ("root_pos_w", "root_quat_w", "root_lin_vel_w", "root_ang_vel_w")


def reference_pins():
    """reference_pins.npz: what the reference's functions return on the inputs of the boundary-case, reset-range,
    two-step pit-command and terrain-lookup tests (tests/test_oracle_edge_cases.py, test_oracle_vs_reference.py,
    test_oracle_neighbours.py), which used to run the robot_lab source at test time.

    Written by running the oracle, not the robot_lab source, on those inputs: the oracle that produced the file is
    unchanged since the commit where the CPU suite ran these very comparisons against the unmodified robot_lab files and
    passed (7096e83: 93 passed, 1 skipped - the variant-library test). Every stored quantity those tests compared
    exactly (commands, reset poses, pit flags, column ranges, terrain masks, the zero pattern of the reward terms) is
    therefore the reference's output bit for bit; the reward values are the reference's to 1e-6 (rtol and atol).
    Reward terms are the reference-owned ones only: those with a reward/ entry in <task>.npz."""
    from oracle import mdp_port as port
    from robot_lab_b200 import terrain as terrain_host
    from robot_lab_b200.cfg import ResetStateCfg, TerrainCfg

    out = {"source": np.array("oracle unchanged since 7096e83, where it matched the robot_lab functions on these inputs")}
    for key in EDGE_KEYS:
        cfg, spec = H.make_spec(key)
        st = H.make_edge_case_state(spec)
        d = port.Derived(st, spec)
        owned = {k[7:] for k in np.load(Path(__file__).resolve().parent / f"{key}.npz").files if k.startswith("reward/")}
        for t in spec.rewards:
            if t.name in owned:
                out[f"edge/{key}/reward/{t.name}"] = port.reward_term(t, st, spec, d).numpy()
        got = port.compute_command(spec, st, {"cmd_uniforms": st["cmd_uniforms"]})
        for k in CMD_KEYS:
            out[f"edge/{key}/command/{k}"] = got[k].numpy()
    for key in RESET_KEYS:
        cfg, spec = H.make_spec(key)
        st, ids, org, u = H.reset_inputs(spec)
        for name, rc in (("default", ResetStateCfg()), ("go2_rough", ResetStateCfg.go2_rough())):
            got = port.reset_scene_state(spec, st, ids, rc, org, u)
            for k in ROOT_KEYS:
                out[f"reset/{key}/{name}/{k}"] = got[k][ids.long()].numpy()
    ter = TerrainCfg(sub_terrains=PIT_SUB_TERRAINS, proportions=PIT_PROPORTIONS)
    for key in PIT_STEP_KEYS:
        cfg, spec = H.make_spec(key)
        n = 2048
        st = make_state(spec, n, seed=21)
        g = torch.Generator().manual_seed(4)
        origins = terrain_host.grid_origins(ter)
        rng = terrain_host.terrain_column_range(ter, "pits")
        was = torch.rand(n, generator=g) < 0.3
        u = st["cmd_uniforms"]
        for it in range(2):
            st["root_pos_w"] = H.pit_positions(n, g)
            got = port.compute_command(spec, st, {"cmd_uniforms": u})
            on = port.is_robot_on_terrain(st["root_pos_w"], origins, rng)
            got.update(port.command_pit_restrict(spec, {**st, **got}, on, was, u))
            for k in CMD_KEYS + ("was_on_pit",):
                out[f"pit_steps/{key}/{it}/{k}"] = got[k].numpy()
            st.update({k: got[k] for k in CMD_KEYS})
            was = got["was_on_pit"]
    _, types, _ = H.terrain_query_inputs(ter)
    for name in RANGE_NAMES:
        rng = terrain_host.terrain_column_range(ter, name)
        out[f"terrain/{name}/column_range"] = np.array(rng if rng is not None else (-1, -1), dtype=np.int64)
        out[f"terrain/{name}/assigned"] = terrain_host.is_env_assigned_to_terrain(ter, types, name).bool().numpy()
    path = Path(__file__).resolve().parent / "reference_pins.npz"
    np.savez_compressed(path, **out)
    print(path.name, path.stat().st_size, "bytes,", len(out), "arrays")


if __name__ == "__main__":
    if "--reference-pins" in sys.argv:
        reference_pins()
    elif "--pits-only" in sys.argv:
        pits()
    else:
        if "--reset-event-only" not in sys.argv:
            main()
        reset_event()
        pits()
