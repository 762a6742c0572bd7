"""Thin object wrapper over the C-ABI: one ``MdpStepEngine`` = one ``RlCtx`` on one GPU.

Every method is a single ``extern "C"`` call with raw device pointers taken from the torch tensors in
``StateBuffers``; launches are asynchronous on torch's current stream (so they compose with CUDA graphs and
with NCCL work enqueued by ``torch.distributed``). No method synchronises.
"""

from __future__ import annotations

import ctypes as C

import torch

from . import _native as nat
from .spec import RewardTermSpec, StepSpec, reward_term_to_ctypes
from .state import StateBuffers


class MdpStepEngine:
    def __init__(self, spec: StepSpec, device: torch.device | str = "cuda:0"):
        self.lib = nat.load()  # raises if the CUDA library is missing: there is no CPU fallback
        self.spec = spec
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise nat.NativeError("the MDP step runs on CUDA devices only")
        self._cspec = spec.to_ctypes()
        self._ctx = C.c_void_p()
        self._pinned_stream = None
        self._has_vel_targets = spec.action.kind is not None and any(spec.action.kind)
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        nat.check(self.lib.rl_ctx_create(C.byref(self._cspec), idx, C.byref(self._ctx)))

    def close(self) -> None:
        if getattr(self, "_ctx", None) is not None and self._ctx.value:
            self.lib.rl_ctx_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self) -> int:
        if self._pinned_stream is not None:   # set for the duration of one env step by ``pinned_stream``
            return self._pinned_stream
        return torch.cuda.current_stream(self.device).cuda_stream

    def pin_stream(self) -> None:
        """Look torch's current stream up once and use it for the following calls (an env step is three launches: the
        lookup costs as much host time as the rest of a call). ``unpin_stream`` ends it."""
        self._pinned_stream = torch.cuda.current_stream(self.device).cuda_stream

    def unpin_stream(self) -> None:
        self._pinned_stream = None

    def set_launch_config(self, warps_per_cta: int = 0, envs_per_cta: int = 0) -> None:
        """Warps per tile of the general kernel (4, 8, 16); envs per CTA is 32 (one lane per env)."""
        nat.check(self.lib.rl_ctx_set_launch_config(self._ctx, envs_per_cta, warps_per_cta))

    def launch_config(self) -> dict:
        """The launch configuration of the general kernel: ``{"envs_per_cta": 32, "warps_per_tile": 4 | 8 | 16}``."""
        epc, nw = C.c_int(0), C.c_int(0)
        nat.check(self.lib.rl_ctx_get_launch_config(self._ctx, C.byref(epc), C.byref(nw)))
        return {"envs_per_cta": epc.value, "warps_per_tile": nw.value}

    def cluster_config(self, num_envs: int) -> dict:
        """What ``step_pre_reset`` / ``step_post_reset`` of ``num_envs`` envs run: cluster size C, tiles per CTA G and warps
        per CTA of the kernels of csrc/mdp_step_v2.cu (C = 0: the general kernel), and the launches they handled so far."""
        c, g, w, n = C.c_int32(0), C.c_int32(0), C.c_int32(0), C.c_int64(0)
        nat.check(self.lib.rl_ctx_get_cluster_config(self._ctx, int(num_envs), C.byref(c), C.byref(g), C.byref(w), C.byref(n)))
        return {"cluster_size": c.value, "tiles_per_cta": g.value, "warps_per_cta": w.value, "launches": n.value}

    def set_pdl(self, enabled: bool) -> None:
        """Programmatic dependent launch between consecutive kernels of this context (launch-latency overlap)."""
        nat.check(self.lib.rl_ctx_set_pdl(self._ctx, int(enabled)))

    def set_debug_buffer(self, buf: torch.Tensor | None) -> None:
        """int64 [ceil(N/32), RL_DEBUG_STRIDE] device tensor receiving per-CTA clock64 stamps (phases, tasks)."""
        nat.check(self.lib.rl_ctx_set_debug_buffer(self._ctx, nat.ptr_of(buf)))

    def schedule(self) -> list[dict]:
        """The static work schedule of the current launch config (see rl_ctx_get_schedule)."""
        out = (C.c_int32 * (nat.RL_MAX_TASKS * 8))()
        n = C.c_int32(0)
        nat.check(self.lib.rl_ctx_get_schedule(self._ctx, out, C.byref(n)))
        keys = ("kind", "a", "b", "owner", "lo", "hi", "col0", "late")
        return [dict(zip(keys, out[i * 8:i * 8 + 8])) for i in range(n.value)]

    def new_buffers(self, num_envs: int, layout: str = "soa") -> StateBuffers:
        return StateBuffers(self.spec, num_envs, self.device, layout)

    def reset_scene_state(self, b: StateBuffers, cfg, env_origins: torch.Tensor | None = None,
                          env_ids: torch.Tensor | None = None, n_env_ids: torch.Tensor | None = None,
                          uniforms: torch.Tensor | None = None, seed: int = 0, step: int = 0, env_id_offset: int = 0,
                          use_step_counter: bool = False, assigned_to_pits: torch.Tensor | None = None) -> None:
        """``reset_root_state_uniform`` (V/mdp/events.py:205-271) + ``reset_joints_by_scale`` [IL] for the env ids, or -
        without ids - for the envs flagged by the last ``step_pre_reset``. ``cfg`` is a ``cfg.ResetStateCfg``;
        ``assigned_to_pits`` (uint8 [N], ``terrain.is_env_assigned_to_terrain``) selects the pit branch (:232-244)."""
        c = nat.RlResetStateCfg()
        drs = [0.0, 0.0, self.spec.layout.asset.init_root_height, 1.0, 0.0, 0.0, 0.0] + [0.0] * 6
        for i, v in enumerate(drs):
            c.default_root_state[i] = v
        for i, k in enumerate(("x", "y", "z", "roll", "pitch", "yaw")):
            c.pose_lo[i], c.pose_hi[i] = cfg.pose_range.get(k, (0.0, 0.0))
            c.vel_lo[i], c.vel_hi[i] = cfg.velocity_range.get(k, (0.0, 0.0))
        c.joint_pos_scale_lo, c.joint_pos_scale_hi = cfg.joint_position_range
        c.joint_vel_scale_lo, c.joint_vel_scale_hi = cfg.joint_velocity_range
        st = b.state_view()
        rnd = b.random(seed, step, env_id_offset, False, use_step_counter)
        org = None
        if env_origins is not None:
            org = nat.RlField(env_origins.data_ptr(), env_origins.stride(0), env_origins.stride(1))
        nat.check(self.lib.rl_reset_scene_state(
            self._ctx, b.N, C.byref(c), C.byref(org) if org is not None else None, C.byref(st),
            b.terminated.data_ptr(), b.truncated.data_ptr(), nat.ptr_of(env_ids), nat.ptr_of(n_env_ids), C.byref(rnd),
            nat.ptr_of(uniforms), nat.ptr_of(assigned_to_pits), self._stream()))

    # ---- neighbours of the path (SURVEY.md 8(f) rows 3, 4) -------------------------------------------------------
    def actuator_cfg(self) -> nat.RlActuatorCfg:
        """RlActuatorCfg of the task's robot (``RobotAsset.actuators``; assets/unitree.py:55-63, 107-115, 504-621)."""
        if getattr(self, "_act_cfg", None) is None:
            tab = self.spec.layout.asset.actuator_table()
            c = nat.RlActuatorCfg()
            c.num_joints = self.spec.J
            for j in range(self.spec.J):
                c.type[j] = nat.ACTUATOR_TYPES[tab["kind"][j]]
                c.stiffness[j], c.damping[j] = tab["stiffness"][j], tab["damping"][j]
                c.effort_limit[j], c.saturation_effort[j] = tab["effort_limit"][j], tab["saturation_effort"][j]
                c.velocity_limit[j] = tab["velocity_limit"][j]
            self._act_cfg = c
        return self._act_cfg

    def actuator_step(self, b: StateBuffers, computed_torque: torch.Tensor | None = None,
                      joint_vel_target: torch.Tensor | None = None, joint_effort_target: torch.Tensor | None = None) -> None:
        """Articulation._apply_actuator_model [IL] for one physics sub-step: reads ``joint_target`` (written by
        ``process_action``), ``joint_pos``, ``joint_vel``; writes ``applied_torque`` (+ ``computed_torque`` [J, N] /
        [N, J] in the buffers' layout when given)."""
        tgt = b.field("joint_target")
        st = b.state_view()
        lay = b.layout
        opt = lambda t: C.byref(nat.field_of(t, lay)) if t is not None else None  # noqa: E731
        vt = opt(joint_vel_target)
        if vt is None and self.spec.action.kind is not None and any(self.spec.action.kind):
            vt = C.byref(b.field("joint_vel_target"))   # the velocity columns of the action (wheels)
        nat.check(self.lib.rl_actuator_step(self._ctx, b.N, C.byref(self.actuator_cfg()), C.byref(tgt), vt,
                                            opt(joint_effort_target), C.byref(st), opt(computed_torque), self._stream()))

    def is_robot_on_terrain(self, b: StateBuffers, grid, out: torch.Tensor | None = None) -> torch.Tensor:
        """``is_robot_on_terrain`` (V/mdp/utils.py:73-127) -> uint8 [N]; ``grid`` is a ``terrain.TerrainGridBuffers``."""
        if out is None:
            out = torch.empty(b.N, dtype=torch.uint8, device=self.device)
        pos = b.field("root_pos_w")
        g = grid.to_ctypes()
        nat.check(self.lib.rl_is_robot_on_terrain(self._ctx, b.N, C.byref(pos), C.byref(g), out.data_ptr(), self._stream()))
        return out

    def command_pit_restrict(self, b: StateBuffers, grid, was_on_pit: torch.Tensor, seed: int = 0, step: int = 0,
                             env_id_offset: int = 0, use_random_inputs: bool = True, use_step_counter: bool = False) -> None:
        """Tail of ``UniformThresholdVelocityCommand._update_command`` (V/mdp/commands.py:61-85): launch it between
        ``step(RESET | COMMAND)`` and ``step(OBS)`` when the terrain has a "pits" sub-terrain."""
        pos = b.field("root_pos_w")
        g = grid.to_ctypes()
        mdp = b.mdp_state()
        rnd = b.random(seed, step, env_id_offset, use_random_inputs, use_step_counter)
        nat.check(self.lib.rl_command_pit_restrict(self._ctx, b.N, C.byref(pos), C.byref(g), C.byref(mdp),
                                                   was_on_pit.data_ptr(), C.byref(rnd), self._stream()))

    def height_scan_cast(self, b: StateBuffers, hf) -> None:
        """Grid-pattern RayCaster [IL] over a height field (``terrain.HeightFieldBuffers``): writes ``ray_hits_z`` and
        ``ray_sensor_pos_z`` of the buffers from ``root_pos_w`` / ``root_quat_w``."""
        st = b.state_view()
        h = hf.to_ctypes()
        nat.check(self.lib.rl_height_scan_cast(self._ctx, b.N, C.byref(h), C.byref(st), self._stream()))

    def contact_sensor_update(self, b: StateBuffers, net_forces_w: torch.Tensor, dt: float, force_threshold: float = 1.0,
                              ring_slot: int = -1) -> None:
        """ContactSensor._update_buffers_impl [IL] for one physics sub-step: history roll (or ring-slot write) and the
        air / contact timers. ``net_forces_w`` is ``[N, B, 3]`` in the history body space."""
        spec = self.spec
        names_h = list(spec.layout.hist_body_names)
        t2h = (C.c_int32 * max(1, spec.Bt))(*[names_h.index(n) for n in spec.layout.time_body_names])
        nf = net_forces_w.reshape(b.N, -1)
        fld = nat.RlField(nf.data_ptr(), nf.stride(0), nf.stride(1) if nf.shape[1] > 1 else 1)
        st = b.state_view()
        nat.check(self.lib.rl_contact_sensor_update(self._ctx, b.N, C.byref(fld), C.byref(st), t2h, float(dt),
                                                    float(force_threshold), int(ring_slot), self._stream()))

    # ---- stage 8 of the step: the interval push event ----------------------------------------------------------
    @staticmethod
    def interval_event_cfg(term) -> nat.RlIntervalEventCfg:
        """RlIntervalEventCfg of an interval ``push_by_setting_velocity`` term (``cfg.EventTermCfg``); a velocity key the
        term does not name is the range (0, 0), as in push_by_setting_velocity [IL]."""
        c = nat.RlIntervalEventCfg()
        c.interval_lo, c.interval_hi = term.interval_range_s
        vr = term.params.get("velocity_range", {})
        for i, k in enumerate(("x", "y", "z", "roll", "pitch", "yaw")):
            c.vel_lo[i], c.vel_hi[i] = vr.get(k, (0.0, 0.0))
        return c

    def interval_push(self, b: StateBuffers, cfg: nat.RlIntervalEventCfg, time_left: torch.Tensor,
                      pushed_ids: torch.Tensor | None = None, n_pushed: torch.Tensor | None = None,
                      env_ids: torch.Tensor | None = None, n_env_ids: torch.Tensor | None = None,
                      dt: float | None = None, uniforms: torch.Tensor | None = None, seed: int = 0, step: int = 0,
                      env_id_offset: int = 0, use_step_counter: bool = False) -> None:
        """EventManager.reset(env_ids) [IL] with ``env_ids`` (timers of those envs resampled), otherwise
        EventManager.apply("interval", dt) [IL] for the step just taken: timers of the envs the last ``step_pre_reset``
        flagged done are resampled, every timer counts down ``dt`` (default: the spec's step_dt), the envs whose timer
        ran out get ``root_lin_vel_w`` / ``root_ang_vel_w`` += U(velocity_range) and their ids land in
        ``pushed_ids[:n_pushed]`` (int32 device tensors [N] / [1]). ``uniforms``: [8, N] U[0,1) instead of Philox."""
        st = b.state_view()
        rnd = b.random(seed, step, env_id_offset, False, use_step_counter)
        dt = self.spec.step_dt if dt is None else dt
        nat.check(self.lib.rl_interval_push(
            self._ctx, b.N, C.byref(cfg), float(dt), time_left.data_ptr(), C.byref(st), b.terminated.data_ptr(),
            b.truncated.data_ptr(), nat.ptr_of(env_ids), nat.ptr_of(n_env_ids), nat.ptr_of(pushed_ids),
            nat.ptr_of(n_pushed), C.byref(rnd), nat.ptr_of(uniforms), self._stream()))

    def reobserve(self, b: StateBuffers, env_ids: torch.Tensor, n_env_ids: torch.Tensor, **rng) -> None:
        """The observation groups again for ``env_ids[:n_env_ids]`` only (the envs an interval push changed after the
        fused post-reset launch observed them): the same rows a full observation pass would write."""
        self.step(b, phases=nat.PHASE_OBS, env_ids=env_ids, n_env_ids=n_env_ids, **rng)

    # ---- the five entry points ----------------------------------------------------------------------
    def process_action(self, b: StateBuffers, with_target: bool = True, advance_step_counter: bool = True,
                       new_action: torch.Tensor | None = None) -> None:
        """``new_action``: the policy's ``[N, A]`` fp32 device tensor, read in place (no copy into the buffers' own
        ``new_action`` field, which is used when this is None)."""
        na = b.field("new_action") if new_action is None else nat.RlField(new_action.data_ptr(), new_action.stride(0), new_action.stride(1))
        mdp = b.mdp_state()
        tgt = b.field("joint_target") if with_target else nat.RlField(None, 0, 0)
        has_vel = with_target and self._has_vel_targets
        vtgt = b.field("joint_vel_target") if has_vel else nat.RlField(None, 0, 0)
        ctr = b.step_counter.data_ptr() if advance_step_counter else None
        nat.check(self.lib.rl_process_action(self._ctx, b.N, C.byref(na), C.byref(mdp), C.byref(tgt), C.byref(vtgt), ctr,
                                             self._stream()))

    def step(self, b: StateBuffers, phases: int = nat.PHASE_ALL, seed: int = 0, step: int = 0, env_id_offset: int = 0,
             use_random_inputs: bool = True, env_ids: torch.Tensor | None = None,
             n_env_ids: torch.Tensor | None = None, use_step_counter: bool = False) -> None:
        st, mdp, out = b.state_view(), b.mdp_state(), b.step_out()
        rnd = b.random(seed, step, env_id_offset, use_random_inputs, use_step_counter)
        nat.check(self.lib.rl_step(self._ctx, b.N, C.byref(st), C.byref(mdp), C.byref(out), C.byref(rnd), phases,
                                   nat.ptr_of(env_ids), nat.ptr_of(n_env_ids), self._stream()))

    def reset_envs(self, b: StateBuffers, env_ids: torch.Tensor, n_env_ids: torch.Tensor, seed: int = 0, step: int = 0,
                   env_id_offset: int = 0, use_random_inputs: bool = True, with_log: bool = True) -> None:
        mdp = b.mdp_state()
        rnd = b.random(seed, step, env_id_offset, use_random_inputs)
        log = b.reset_log() if with_log else nat.RlResetLog()
        nat.check(self.lib.rl_reset_envs(self._ctx, b.N, C.byref(mdp), b.done_bits.data_ptr(), C.byref(rnd), C.byref(log),
                                         nat.ptr_of(env_ids), nat.ptr_of(n_env_ids), self._stream()))

    def post_reset(self, b: StateBuffers, seed: int = 0, step: int = 0, env_id_offset: int = 0,
                   use_random_inputs: bool = True, use_step_counter: bool = False) -> None:
        """Everything ManagerBasedRLEnv.step() [IL] does for the reset ids after the external (physics) reset,
        in one launch: manager reset + logging means, command.compute, both observation groups."""
        self.step(b, phases=nat.PHASE_RESET | nat.PHASE_COMMAND | nat.PHASE_OBS, seed=seed, step=step,
                  env_id_offset=env_id_offset, use_random_inputs=use_random_inputs, env_ids=b.reset_ids,
                  n_env_ids=b.n_reset, use_step_counter=use_step_counter)

    # ---- the env step as two launches around the external reset (the reference's exact order) ---------------
    PRE_RESET = nat.PHASE_DONES | nat.PHASE_REWARDS | nat.PHASE_COMPACT
    POST_RESET = nat.PHASE_RESET | nat.PHASE_COMMAND | nat.PHASE_OBS

    def step_pre_reset(self, b: StateBuffers, **rng) -> None:
        """termination terms, reward terms (+ sums / step reward), reset-id compaction: what ManagerBasedRLEnv.step()
        [IL] evaluates before ``_reset_idx``."""
        self.step(b, phases=self.PRE_RESET, **rng)

    def step_post_reset(self, b: StateBuffers, **rng) -> None:
        """Manager reset (+ logging means) of the envs flagged done by ``step_pre_reset``, then command.compute and
        both observation groups for ALL envs - full tiles, no gather."""
        self.step(b, phases=self.POST_RESET, **rng)

    def term_eval(self, term: RewardTermSpec, b: StateBuffers, out: torch.Tensor | None = None,
                  terminated: torch.Tensor | None = None) -> torch.Tensor:
        if out is None:
            out = torch.empty(b.N, device=self.device)
        ct = reward_term_to_ctypes(term)
        st, mdp = b.state_view(), b.mdp_state()
        nat.check(self.lib.rl_term_eval(self._ctx, b.N, C.byref(ct), C.byref(st), C.byref(mdp), nat.ptr_of(terminated),
                                        out.data_ptr(), self._stream()))
        return out
