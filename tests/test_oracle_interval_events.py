"""The interval push event (stage 8 of ManagerBasedRLEnv.step() [IL]: event_manager.apply("interval") with
push_by_setting_velocity, the reference's randomize_push_robot at V/velocity_env_cfg.py:366-371) on the CPU: the oracle
against a scalar, step-by-step re-derivation of the IsaacLab rules, and the cfg surface. No GPU needed.
PARITY UNPINNED like every [IL] piece: IsaacLab is not vendored, the rules are restated from the upstream algorithm."""

import numpy as np
import pytest
import torch

import interval_events_oracle as IO
from oracle import philox

F = np.float32


def _scalar_steps(t0, lo, hi, dt, u_fire, steps):
    """One env, fp32 scalar arithmetic: time_left -= dt; fire = time_left < 1e-6 -> resample. Returns the fire steps."""
    t, fired = F(t0), []
    for k in range(steps):
        t = F(t - F(dt))
        if t < F(1e-6):
            t = F(F(F(u_fire) * F(F(hi) - F(lo))) + F(lo))
            fired.append(k)
    return fired, t


@pytest.mark.parametrize("period,dt,k", [(1.0, 0.02, 50), (0.3, 0.1, 3), (2.0, 0.02, 101)])
def test_constant_interval_fires_every_kth_step_and_matches_the_scalar_rederivation(period, dt, k):
    # lo == hi: after every push the timer is exactly `period` again, so an env fires every k-th step. k is what fp32
    # `time_left -= dt` gives: 1.0 s at dt 0.02 leaves +3.9e-7 after 50 decrements - below the 1e-6 threshold, so it
    # fires at 50 (a `<= 0` test would wait for 51); 2.0 s leaves +1.3e-6 after 100 and fires at 101.
    n, steps = 16, 3 * k + 2
    time_left = torch.full((n,), period, dtype=torch.float32)
    lin, ang = torch.zeros(n, 3), torch.zeros(n, 3)
    vr = {"x": (-0.5, 0.5), "y": (-0.5, 0.5)}
    g = torch.Generator().manual_seed(3)
    fires = []
    for _ in range(steps):
        u = torch.rand(8, n, generator=g)
        out = IO.interval_push(time_left, lin, ang, (period, period), vr, dt, u, reset=torch.zeros(n, dtype=torch.bool))
        time_left, lin, ang = out["time_left"], out["root_lin_vel_w"], out["root_ang_vel_w"]
        fires.append(out["pushed"].clone())
    fires = torch.stack(fires)                                            # [steps, n]
    expect, t_end = _scalar_steps(period, period, period, dt, 0.25, steps)
    assert expect == [k - 1, 2 * k - 1, 3 * k - 1]
    for e in range(n):
        assert fires[:, e].nonzero().flatten().tolist() == expect
    assert torch.all(time_left == torch.tensor(t_end))
    if period == 1.0:   # the threshold at work: the residue at step k is positive and below 1e-6
        t = F(period)
        for _ in range(k):
            t = F(t - F(dt))
        assert F(0.0) < t < F(1e-6)


def test_scalar_rederivation_with_resets_and_pushes_matches_the_oracle():
    n, steps, dt, lo, hi = 64, 300, 0.02, 0.5, 1.5
    vr = {"x": (-0.5, 0.5), "y": (-0.25, 0.75), "yaw": (-1.0, 1.0)}
    g = torch.Generator().manual_seed(11)
    time_left = torch.rand(n, generator=g) * (hi - lo) + lo
    lin, ang = torch.randn(n, 3, generator=g), torch.randn(n, 3, generator=g)
    t_s = time_left.numpy().astype(F).copy()
    v_s = torch.cat([lin, ang], 1).numpy().astype(F).copy()
    keys = IO.VELOCITY_KEYS
    for _ in range(steps):
        u = torch.rand(8, n, generator=g)
        reset = torch.rand(n, generator=g) < 0.05
        out = IO.interval_push(time_left, lin, ang, (lo, hi), vr, dt, u, reset=reset)
        un = u.numpy()
        for e in range(n):   # scalar restatement, one env at a time
            t = t_s[e]
            if reset[e]:
                t = F(F(un[0, e] * F(F(hi) - F(lo))) + F(lo))
            t = F(t - F(dt))
            fire = t < F(1e-6)
            if fire:
                t = F(F(un[1, e] * F(F(hi) - F(lo))) + F(lo))
                for q, key in enumerate(keys):
                    a, b = vr.get(key, (0.0, 0.0))
                    v_s[e, q] = F(v_s[e, q] + F(F(un[2 + q, e] * F(F(b) - F(a))) + F(a)))
            t_s[e] = t
            assert bool(out["pushed"][e]) == bool(fire)
        time_left, lin, ang = out["time_left"], out["root_lin_vel_w"], out["root_ang_vel_w"]
        assert np.array_equal(time_left.numpy(), t_s)
        assert np.array_equal(torch.cat([lin, ang], 1).numpy(), v_s)


def test_an_env_reset_in_this_step_is_not_pushed_in_it():
    n = 32
    time_left = torch.full((n,), 1e-7)                                   # every timer would run out this step
    lin, ang = torch.ones(n, 3), torch.ones(n, 3)
    reset = torch.arange(n) % 3 == 0
    u = torch.rand(8, n, generator=torch.Generator().manual_seed(5))
    out = IO.interval_push(time_left, lin, ang, (10.0, 15.0), {"x": (-0.5, 0.5)}, 0.02, u, reset=reset)
    assert torch.equal(out["pushed"], ~reset)
    assert bool(torch.all(out["time_left"][reset] >= 10.0 - 0.02))
    assert torch.equal(out["root_lin_vel_w"][reset], lin[reset])


def test_reset_form_resamples_the_listed_timers_only():
    n = 20
    time_left = torch.full((n,), 3.0)
    lin, ang = torch.zeros(n, 3), torch.zeros(n, 3)
    u = torch.rand(8, n, generator=torch.Generator().manual_seed(1))
    ids = torch.tensor([1, 4, 19], dtype=torch.int32)
    out = IO.interval_push(time_left, lin, ang, (10.0, 15.0), {}, 0.02, u, env_ids=ids)
    want = time_left.clone()
    want[ids.long()] = u[0, ids.long()] * 5.0 + 10.0
    assert torch.equal(out["time_left"], want)
    assert not out["pushed"].any()


def test_missing_velocity_keys_leave_those_components_unchanged():
    n = 50
    g = torch.Generator().manual_seed(2)
    lin, ang = torch.randn(n, 3, generator=g), torch.randn(n, 3, generator=g)
    u = torch.rand(8, n, generator=g)
    out = IO.interval_push(torch.zeros(n), lin, ang, (1.0, 2.0), {"x": (-0.5, 0.5), "pitch": (0.1, 0.2)}, 0.02, u,
                             reset=torch.zeros(n, dtype=torch.bool))
    assert out["pushed"].all()
    assert not torch.equal(out["root_lin_vel_w"][:, 0], lin[:, 0])
    assert not torch.equal(out["root_ang_vel_w"][:, 1], ang[:, 1])
    for q in (1, 2):
        assert torch.equal(out["root_lin_vel_w"][:, q], lin[:, q])
    for q in (0, 2):
        assert torch.equal(out["root_ang_vel_w"][:, q], ang[:, q])


def test_interval_uniform_table_layout():
    u = IO.interval_uniforms(64, seed=9, step=4, env_id_offset=128).numpy()
    assert u.shape == (8, 64)
    ids = np.arange(64)
    assert np.array_equal(u[0], philox.draw(ids, 9, 4, 128, IO.STREAM_INTERVAL_RESET, 0)[:, 0])
    assert np.array_equal(u[1:5].T, philox.draw(ids, 9, 4, 128, IO.STREAM_INTERVAL_PUSH, 0))
    assert np.array_equal(u[5:8].T, philox.draw(ids, 9, 4, 128, IO.STREAM_INTERVAL_PUSH, 1)[:, :3])
    assert IO.STREAM_INTERVAL_RESET > 5 and IO.STREAM_INTERVAL_PUSH < philox.STREAM_OBS
    # the kernel's stream numbers (robot_lab_b200/csrc/rl_common.cuh)
    from pathlib import Path
    import re

    src = (Path(__file__).resolve().parent.parent / "robot_lab_b200" / "csrc" / "rl_common.cuh").read_text()
    streams = {m.group(1): int(m.group(2)) for m in re.finditer(r"RL_STREAM_(\w+) = (\d+)", src)}
    assert streams["INTERVAL_RESET"] == IO.STREAM_INTERVAL_RESET and streams["INTERVAL_PUSH"] == IO.STREAM_INTERVAL_PUSH
    assert streams["PIT_RESAMPLE"] < IO.STREAM_INTERVAL_RESET < IO.STREAM_INTERVAL_PUSH < streams["OBS"]


# ---- cfg surface --------------------------------------------------------------------------------------------------
def test_push_is_off_by_default_and_the_helper_is_the_reference_term():
    from robot_lab_b200 import mdp
    from robot_lab_b200.envs import interval_push_terms
    from robot_lab_b200.tasks import TASKS, make_env_cfg
    from robot_lab_b200.tasks.locomotion_velocity import push_robot_event_term

    for task in TASKS:
        cfg = make_env_cfg(task, num_envs=8)
        assert cfg.events.randomize_push_robot is None, task
        assert interval_push_terms(cfg) == []
    term = push_robot_event_term()
    assert term.func is mdp.push_by_setting_velocity and term.mode == "interval" and not term.is_global_time
    assert term.interval_range_s == (10.0, 15.0)
    assert term.params == {"velocity_range": {"x": (-0.5, 0.5), "y": (-0.5, 0.5)}}
    cfg = make_env_cfg("RobotLab-Isaac-Velocity-Rough-Unitree-Go2-v0", num_envs=8)
    cfg.events.randomize_push_robot = term
    assert interval_push_terms(cfg) == [("randomize_push_robot", term)]
    # the marker is no term of the fused step
    assert "push_by_setting_velocity" not in mdp.all_terms()
    with pytest.raises(NotImplementedError):
        mdp.push_by_setting_velocity(None, None, {})


def test_interval_event_cfg_fills_missing_keys_with_zero_ranges():
    from robot_lab_b200.engine import MdpStepEngine
    from robot_lab_b200.tasks.locomotion_velocity import push_robot_event_term

    c = MdpStepEngine.interval_event_cfg(push_robot_event_term((1.0, 2.0), {"y": (-0.5, 0.25), "yaw": (0.0, 1.0)}))
    assert (c.interval_lo, c.interval_hi) == (1.0, 2.0)
    assert list(c.vel_lo) == [0.0, -0.5, 0.0, 0.0, 0.0, 0.0]
    assert list(c.vel_hi) == [0.0, 0.25, 0.0, 0.0, 0.0, 1.0]


def _bad_cfgs():
    from robot_lab_b200 import mdp
    from robot_lab_b200.cfg import EventTermCfg, RewardTermCfg, SceneEntityCfg

    push = mdp.push_by_setting_velocity
    vr = {"velocity_range": {"x": (-0.5, 0.5)}}
    return {
        "reset_mode": EventTermCfg(func=push, mode="reset", params=vr),
        "startup_mode": EventTermCfg(func=push, mode="startup", params=vr),
        "other_function": EventTermCfg(func=mdp.lin_vel_z_l2, mode="interval", interval_range_s=(1.0, 2.0)),
        "global_time": EventTermCfg(func=push, mode="interval", interval_range_s=(1.0, 2.0), is_global_time=True, params=vr),
        "no_interval": EventTermCfg(func=push, mode="interval", params=vr),
        "lo_above_hi": EventTermCfg(func=push, mode="interval", interval_range_s=(3.0, 2.0), params=vr),
        "bad_velocity_key": EventTermCfg(func=push, mode="interval", interval_range_s=(1.0, 2.0),
                                         params={"velocity_range": {"vx": (-0.5, 0.5)}}),
        "velocity_lo_above_hi": EventTermCfg(func=push, mode="interval", interval_range_s=(1.0, 2.0),
                                             params={"velocity_range": {"x": (0.5, -0.5)}}),
        "other_asset": EventTermCfg(func=push, mode="interval", interval_range_s=(1.0, 2.0),
                                    params={**vr, "asset_cfg": SceneEntityCfg("box")}),
        "extra_param": EventTermCfg(func=push, mode="interval", interval_range_s=(1.0, 2.0), params={**vr, "scale": 2.0}),
        "not_an_event_term": RewardTermCfg(func=push, weight=1.0),
    }


@pytest.mark.parametrize("name", list(_bad_cfgs()))
def test_unsupported_event_terms_raise_naming_the_term(name):
    from robot_lab_b200.envs import interval_push_terms
    from robot_lab_b200.tasks import make_env_cfg

    cfg = make_env_cfg("RobotLab-Isaac-Velocity-Rough-Unitree-Go2-v0", num_envs=8)
    setattr(cfg.events, name, _bad_cfgs()[name])
    with pytest.raises(ValueError, match=name):
        interval_push_terms(cfg)


def test_two_interval_push_terms_raise():
    from robot_lab_b200.envs import interval_push_terms
    from robot_lab_b200.tasks import make_env_cfg
    from robot_lab_b200.tasks.locomotion_velocity import push_robot_event_term

    cfg = make_env_cfg("RobotLab-Isaac-Velocity-Rough-Unitree-Go2-v0", num_envs=8)
    cfg.events.randomize_push_robot = push_robot_event_term()
    cfg.events.second_push = push_robot_event_term()
    with pytest.raises(ValueError, match="second_push"):
        interval_push_terms(cfg)
