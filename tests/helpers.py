"""Shared helpers of the parity tests: build spec / synthetic state / engine, run both sides, compare."""

from __future__ import annotations

import torch

from oracle import mdp_port as port
from robot_lab_b200 import _native as nat
from robot_lab_b200.spec import compact_layout, compile_step_spec
from robot_lab_b200.synthetic import make_state
from robot_lab_b200.tasks import make_env_cfg

# fp32 parity bar of BASELINE.json's north_star: 1e-5 relative. The absolute floor covers outputs whose true
# value is ~0 (sums with cancellation, products with a 0/1 mask): 1e-6 times the O(1) scale of the inputs.
RTOL, ATOL = 1e-5, 1e-6

TASKS = {
    "a1_flat": "RobotLab-Isaac-Velocity-Flat-Unitree-A1-v0",
    "go2_flat": "RobotLab-Isaac-Velocity-Flat-Unitree-Go2-v0",
    "go2_rough": "RobotLab-Isaac-Velocity-Rough-Unitree-Go2-v0",
    "g1_rough": "RobotLab-Isaac-Velocity-Rough-Unitree-G1-v0",
    "g1_rough_37": "RobotLab-Isaac-Velocity-Rough-Unitree-G1-37dof-v0",
    "g1_flat": "RobotLab-Isaac-Velocity-Flat-Unitree-G1-v0",
    "a1_rough": "RobotLab-Isaac-Velocity-Rough-Unitree-A1-v0",
}


def make_spec(task_key: str, full_layout: bool = False):
    cfg = make_env_cfg(TASKS[task_key])
    layout = cfg.scene.make_layout() if full_layout else compact_layout(cfg)
    return cfg, compile_step_spec(cfg, layout)


def rnd_inputs(st: dict) -> dict:
    return {"cmd_uniforms": st["cmd_uniforms"], "obs_uniforms_policy": st["obs_uniforms_policy"],
            "obs_uniforms_critic": st["obs_uniforms_critic"]}


def oracle_step(spec, st, skip_done_envs=False, rnd=None):
    return port.step(spec, st, rnd if rnd is not None else rnd_inputs(st), skip_done_envs=skip_done_envs)


def gpu_step_outputs(b) -> dict:
    """Device outputs of one rl_step call, in the oracle's logical shapes (CPU tensors)."""
    n = int(b.n_reset.item())
    out = {
        "episode_length": b.logical("episode_length").cpu(),
        "terminated": b.terminated.cpu().bool(), "truncated": b.truncated.cpu().bool(),
        "done_bits": b.done_bits.cpu().to(torch.int32),
        "reward": b.reward.cpu(), "episode_sums": b.logical("episode_sums").cpu().contiguous(),
        "step_reward": b.logical("step_reward").cpu().contiguous(), "reset_ids": b.reset_ids[:n].cpu(),
        "command": b.logical("command").cpu().contiguous(), "heading_target": b.logical("heading_target").cpu(),
        "time_left": b.logical("time_left").cpu(), "is_heading_env": b.logical("is_heading_env").cpu(),
        "is_standing_env": b.logical("is_standing_env").cpu(),
        "metric_error_vel_xy": b.logical("metric_error_vel_xy").cpu(),
        "metric_error_vel_yaw": b.logical("metric_error_vel_yaw").cpu(),
    }
    if b.obs[0] is not None:
        out["obs_policy"] = b.obs[0].cpu()
    if b.obs[1] is not None:
        out["obs_critic"] = b.obs[1].cpu()
    return out


EXACT_KEYS = ("episode_length", "terminated", "truncated", "done_bits", "reset_ids", "is_heading_env", "is_standing_env")


def compare_outputs(got: dict, ref: dict, rtol=RTOL, atol=ATOL, keys=None) -> dict:
    """Returns {key: (max_abs_err, n_bad)}; raises AssertionError listing every failing key."""
    report, failures = {}, []
    for k in keys or ref.keys():
        if k not in got:
            continue
        g, r = got[k], ref[k]
        if k in EXACT_KEYS:
            ok = g.shape == r.shape and torch.equal(g.to(r.dtype), r)
            report[k] = (0.0 if ok else float("nan"), 0 if ok else int((g.to(r.dtype) != r).sum()) if g.shape == r.shape else -1)
            if not ok:
                failures.append(f"{k}: exact mismatch ({report[k][1]} elements)")
            continue
        g, r = g.float(), r.float()
        if g.shape != r.shape:
            failures.append(f"{k}: shape {tuple(g.shape)} vs {tuple(r.shape)}")
            continue
        both_inf = torch.isinf(g) & torch.isinf(r) & (g == r)
        err = torch.where(both_inf, torch.zeros_like(g), (g - r).abs())
        bad = err > (atol + rtol * r.abs())
        bad |= torch.isnan(g) != torch.isnan(r)
        report[k] = (float(err[~torch.isnan(err)].max()) if err.numel() else 0.0, int(bad.sum()))
        if bad.any():
            i = int(bad.flatten().nonzero()[0])
            failures.append(f"{k}: {int(bad.sum())} bad, max abs err {report[k][0]:.3e}, first bad flat idx {i}: "
                            f"got {g.flatten()[i].item():.9g} want {r.flatten()[i].item():.9g}")
    if failures:
        raise AssertionError("parity failures:\n  " + "\n  ".join(failures))
    return report


def make_catalogue_spec():
    """Go2 with EVERY reward term of the reference's catalogue switched on (weights 1), incl. the ones the in-scope
    tasks leave at 0 (V/velocity_env_cfg.py:379-644) and feet_distance_xy_exp (commented out there, :633-642)."""
    import math

    from robot_lab_b200 import mdp
    from robot_lab_b200.cfg import RewardTermCfg, SceneEntityCfg
    from robot_lab_b200.spec import SceneLayout
    from robot_lab_b200.tasks.locomotion_velocity import _reward_catalogue

    cfg = make_env_cfg(TASKS["go2_rough"])
    cat = _reward_catalogue()
    foot = [".*_foot"]
    for name in ("feet_air_time", "feet_air_time_variance", "feet_contact", "feet_contact_without_cmd", "feet_stumble",
                 "contact_forces"):
        getattr(cat, name).params["sensor_cfg"].body_names = foot
    cat.undesired_contacts.params["sensor_cfg"].body_names = ["^(?!.*_foot).*"]
    cat.feet_slide.params["sensor_cfg"].body_names = foot
    for name in ("feet_slide", "feet_height", "feet_height_body", "feet_distance_y_exp"):
        getattr(cat, name).params["asset_cfg"].body_names = foot
    cat.feet_distance_y_exp.params["stance_width"] = 0.3
    cat.feet_gait.params["synced_feet_pair_names"] = (("FL_foot", "RR_foot"), ("FR_foot", "RL_foot"))
    cat.base_height_l2.params["sensor_cfg"] = None
    cat.base_height_l2.params["target_height"] = 0.33
    cat.joint_mirror.params["mirror_joints"] = [["FR_(hip|thigh|calf).*", "RL_(hip|thigh|calf).*"],
                                                ["FL_(hip|thigh|calf).*", "RR_(hip|thigh|calf).*"]]
    cat.action_mirror.params["mirror_joints"] = cat.joint_mirror.params["mirror_joints"]
    cat.wheel_vel_penalty.params["asset_cfg"].joint_names = [".*_calf_joint"]
    cat.wheel_vel_penalty.params["sensor_cfg"].body_names = foot
    cat.feet_distance_xy_exp = RewardTermCfg(func=mdp.feet_distance_xy_exp, weight=0.0, params={
        "std": math.sqrt(0.25), "asset_cfg": SceneEntityCfg("robot", body_names=foot), "stance_length": 0.4,
        "stance_width": 0.3})
    cat.joint_deviation_hip = RewardTermCfg(func=mdp.joint_deviation_l1, weight=0.0, params={
        "asset_cfg": SceneEntityCfg("robot", joint_names=[".*_hip_joint"])})
    for _, term in cat.items():
        term.weight = 1.0
    cfg.rewards = cat
    full = cfg.scene.make_layout()
    feet = tuple(n for n in full.asset.body_names if n.endswith("_foot"))
    layout = SceneLayout(full.asset, full.hist_body_names, feet, feet, full.terrain, full.num_rays, full.hist_len)
    return cfg, compile_step_spec(cfg, layout)


def oracle_env_rollout(spec, mdp0: dict, phys: list[dict], actions: list[torch.Tensor], seed: int, n_envs: int):
    """CPU replay of ``ManagerBasedRLEnv.step()`` (robot_lab_b200.envs) for a list of physics states / actions, with
    the production Philox streams: returns per-step (obs_policy, obs_critic, reward, terminated, truncated, mdp)."""
    mdp = {k: v.clone() for k, v in mdp0.items()}
    outs = []
    keys_cmd = ("command", "heading_target", "time_left", "is_heading_env", "is_standing_env",
                "metric_error_vel_xy", "metric_error_vel_yaw")
    for t, (ph, act) in enumerate(zip(phys, actions)):
        rnd = {"seed": seed, "step": t + 1, "env_id_offset": 0}
        action, prev, _ = port.process_action(spec, mdp, act)
        mdp["action"], mdp["prev_action"] = action, prev
        st = {**ph, **mdp}
        out = port.step(spec, st, rnd, skip_done_envs=True)
        for k in keys_cmd + ("episode_length", "episode_sums"):
            mdp[k] = out[k]
        st = {**ph, **mdp}
        st2, _log = port.reset_envs(spec, st, out["reset_ids"], out["done_bits"], rnd)
        mdp.update(st2)
        mask = torch.zeros(n_envs, dtype=torch.bool)
        mask[out["reset_ids"].long()] = True
        st = {**ph, **mdp}
        mdp.update(port.compute_command(spec, st, rnd, active=mask))
        st = {**ph, **mdp}
        obs_p = torch.where(mask[:, None], port.compute_obs_group(spec, 0, st, rnd), out["obs_policy"])
        obs_c = torch.where(mask[:, None], port.compute_obs_group(spec, 1, st, rnd), out["obs_critic"])
        outs.append({"obs_policy": obs_p, "obs_critic": obs_c, "reward": out["reward"], "terminated": out["terminated"],
                     "truncated": out["truncated"], "mdp": {k: v.clone() for k, v in mdp.items()}})
    return outs


def make_edge_case_state(spec, n: int = 64, seed: int = 4321) -> dict:
    """Synthetic state whose first envs sit exactly ON the decision boundaries of the path (SURVEY.md section 4, item 3):
    upright / inverted / sideways base (gate 1, 0, 0), zero and threshold-norm commands, contact forces of exactly the
    1 N / 100 N thresholds, +-inf ray hits, episode length one step before / at the time-out, root position exactly on
    the terrain bound, contact / air timers exactly at step_dt and at the 0.5 s threshold, joints exactly on their
    soft limits. The remaining envs keep the ordinary synthetic values (Go2 body layout assumed)."""
    st = make_state(spec, n, seed=seed)
    names = list(spec.layout.hist_body_names)
    foot, calf = names.index("FL_foot"), names.index("FL_calf")
    inf = float("inf")
    q = st["root_quat_w"]
    q[0] = torch.tensor([1.0, 0.0, 0.0, 0.0])                     # upright: gate 1
    q[1] = torch.tensor([0.0, 1.0, 0.0, 0.0])                     # upside down: gate 0
    q[2] = torch.tensor([0.5 ** 0.5, 0.5 ** 0.5, 0.0, 0.0])       # 90 deg roll: projected gravity z ~ 0
    for e in (0, 1, 2):
        st["root_lin_vel_w"][e] = 0.0
        st["root_ang_vel_w"][e] = 0.0
    st["command"][0] = 0.0                                        # standing still
    st["command"][3] = torch.tensor([0.1, 0.0, 0.0])              # |cmd| == 0.1: strict comparisons on both sides
    st["command"][4] = torch.tensor([0.06, 0.08, 0.0])            # |cmd| == 0.1 up to rounding
    h = st["net_forces_w_history"]
    h[5] = 0.0
    h[5, 1, calf] = torch.tensor([1.0, 0.0, 0.0])                 # |F| == 1.0: NOT an undesired contact (strict >)
    h[5, 2, foot] = torch.tensor([0.0, 0.0, 100.0])               # |F| == 100: contact_forces adds exactly 0
    h[6] = 0.0
    h[6, 0, calf] = torch.tensor([0.6, 0.8, 0.0])                 # 1.0 up to rounding
    st["ray_hits_z"][7] = inf                                     # every ray misses: height scan clips to -1
    st["ray_hits_z"][8] = -inf
    st["ray_hits_z"][9, ::2] = inf
    st["episode_length"][10] = spec.max_episode_length - 2        # 998 -> 999: no time-out
    st["episode_length"][11] = spec.max_episode_length - 1        # 999 -> 1000: time-out
    bound = [d.p for d in spec.dones if d.type_name == "terrain_out_of_bounds"]
    if bound:
        st["root_pos_w"][12, 0] = bound[0][0]                     # |x| == bound: strict >, stays in
        st["root_pos_w"][12, 1] = 0.0
        st["root_pos_w"][13, 0] = 0.0
        st["root_pos_w"][13, 1] = -bound[0][1] - 1e-3             # just outside in y
    dt = float(spec.step_dt)
    st["current_contact_time"][14] = dt                           # first contact exactly one step ago
    st["current_air_time"][14] = 0.0
    st["last_air_time"][14] = 0.5                                 # feet_air_time: (last_air - 0.5) == 0
    st["last_contact_time"][14] = 0.5
    st["command"][14] = torch.tensor([0.5, 0.0, 0.0])
    lims = torch.tensor(spec.layout.asset.soft_joint_pos_limits(), dtype=torch.float32)   # [J, 2]
    st["joint_pos"][15] = lims[:, 0]                              # exactly on the lower soft limits: violation 0
    st["joint_pos"][16] = lims[:, 1]                              # ... and on the upper ones
    return st


# ---- inputs of the tests pinned by tests/golden/reference_pins.npz (make_golden.py::reference_pins) ----------------
def reference_pins() -> dict:
    import numpy as np
    from pathlib import Path

    z = np.load(Path(__file__).resolve().parent / "golden" / "reference_pins.npz")
    return {k: torch.from_numpy(z[k]) for k in z.files if k != "source"}


def reset_inputs(spec):
    """80 envs, uniforms / env origins from seed 11, six reset ids."""
    n = 80
    st = make_state(spec, n)
    g = torch.Generator().manual_seed(11)
    u = torch.rand(12 + 2 * spec.J, n, generator=g)
    org = torch.randn(n, 3, generator=g) * 15.0
    return st, torch.tensor([0, 3, 4, 17, 42, 79], dtype=torch.int32), org, u


def pit_positions(n, g):
    return torch.stack([(torch.rand(n, generator=g) - 0.5) * 70.0, (torch.rand(n, generator=g) - 0.5) * 150.0,
                        torch.rand(n, generator=g)], dim=1)


def terrain_query_inputs(ter_cfg):
    """4096 robots spread over a generator terrain with a "pits" sub-terrain, random sub-terrain types (seed 3)."""
    from robot_lab_b200 import terrain as terrain_host

    n = 4096
    g = torch.Generator().manual_seed(3)
    pos = torch.stack([(torch.rand(n, generator=g) - 0.5) * 100.0, (torch.rand(n, generator=g) - 0.5) * 190.0,
                       torch.rand(n, generator=g)], dim=1)
    types = torch.randint(0, ter_cfg.num_cols, (n,), generator=g)
    origins = terrain_host.grid_origins(ter_cfg)
    origins[:, :, 2] = torch.rand(origins.shape[:2], generator=g)
    return pos, types, origins
