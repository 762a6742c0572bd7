"""Oracle of the interval push event (rl_interval_push, stage 8 of the env step): a restatement in eager fp32 PyTorch,
and the kernel's two Philox streams in the counter layout of ``oracle/philox.py``.

TEST INFRASTRUCTURE, like ``oracle/``: only the tests and tools import it. It sits next to the tests, which use it,
rather than in ``oracle/``, whose pinned modules are left as they are.
"""

from __future__ import annotations

import numpy as np
import torch

from oracle import philox

# rl_interval_push draws from the two streams after RL_STREAM_PIT_RESAMPLE (5) in robot_lab_b200/csrc/rl_common.cuh
STREAM_INTERVAL_RESET = 6   # interval timer drawn on reset (x of block 0)
STREAM_INTERVAL_PUSH = 7    # interval timer drawn on fire (x of block 0), push velocities (y, z, w of block 0, x, y, z of block 1)


def interval_uniforms(n: int, seed: int, step: int, env_id_offset: int) -> torch.Tensor:
    """[8, N] table of rl_interval_push: timer on reset, timer on fire, velocity x, y, z, roll, pitch, yaw."""
    ids = np.arange(n)
    r = philox.draw(ids, seed, step, env_id_offset, STREAM_INTERVAL_RESET, 0)
    a = philox.draw(ids, seed, step, env_id_offset, STREAM_INTERVAL_PUSH, 0)
    b = philox.draw(ids, seed, step, env_id_offset, STREAM_INTERVAL_PUSH, 1)
    u = np.concatenate([r[:, :1], a, b[:, :3]], axis=1).T.copy()
    return torch.from_numpy(u)


VELOCITY_KEYS = ("x", "y", "z", "roll", "pitch", "yaw")


def interval_push(time_left: torch.Tensor, root_lin_vel_w: torch.Tensor, root_ang_vel_w: torch.Tensor,
                  interval_range_s: tuple[float, float], velocity_range: dict, dt: float, uniforms: torch.Tensor,
                  reset: torch.Tensor | None = None, env_ids: torch.Tensor | None = None) -> dict:
    """EventManager.reset / apply("interval") [IL] (isaaclab/managers/event_manager.py: _prepare_terms, reset, apply) for
    one non-global interval term whose function is push_by_setting_velocity [IL] (isaaclab/envs/mdp/events.py) - the
    reference's randomize_push_robot (V/velocity_env_cfg.py:366-371). PARITY UNPINNED: IsaacLab is not vendored;
    restated from the upstream algorithm.

    ``uniforms`` is the [8, N] U[0,1) table: row 0 timer on reset, row 1 timer on fire, rows 2-7 velocity x, y, z, roll,
    pitch, yaw. With ``env_ids`` (EventManager.reset): time_left[env_ids] = rand * (hi - lo) + lo, nothing else. Without
    (the step form): envs in the bool mask ``reset`` get that fresh timer first (the reset at stage 6), then
        time_left -= dt;  fire = time_left < 1e-6;  time_left[fire] = rand * (hi - lo) + lo
        root_vel_w[fire] += sample_uniform(lo, hi)      (root_vel_w = lin x, y, z, ang x, y, z; missing keys (0, 0))
    Returns time_left, root_lin_vel_w, root_ang_vel_w and ``pushed`` (bool [N])."""
    f32 = torch.float32
    lo, hi = torch.tensor(interval_range_s[0], dtype=f32), torch.tensor(interval_range_s[1], dtype=f32)
    t = time_left.clone()
    lin, ang = root_lin_vel_w.clone(), root_ang_vel_w.clone()
    n = t.shape[0]
    if env_ids is not None:
        ids = env_ids.long()
        t[ids] = uniforms[0, ids] * (hi - lo) + lo
        return {"time_left": t, "root_lin_vel_w": lin, "root_ang_vel_w": ang, "pushed": torch.zeros(n, dtype=torch.bool)}
    if reset is not None:
        r = reset.nonzero(as_tuple=False).flatten()
        t[r] = uniforms[0, r] * (hi - lo) + lo
    t -= torch.tensor(dt, dtype=f32)
    fire = t < 1e-6
    ids = fire.nonzero(as_tuple=False).flatten()
    if len(ids) > 0:
        t[ids] = uniforms[1, ids] * (hi - lo) + lo
        ranges = torch.tensor([velocity_range.get(k, (0.0, 0.0)) for k in VELOCITY_KEYS], dtype=f32)
        vel_w = torch.cat([lin[ids], ang[ids]], dim=1)
        vel_w += uniforms[2:8, ids].t() * (ranges[:, 1] - ranges[:, 0]) + ranges[:, 0]
        lin[ids] = vel_w[:, 0:3]
        ang[ids] = vel_w[:, 3:6]
    return {"time_left": t, "root_lin_vel_w": lin, "root_ang_vel_w": ang, "pushed": fire}
