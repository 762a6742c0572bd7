"""The interval push event on a GPU (stage 8 of ManagerBasedRLEnv.step() [IL], the reference's randomize_push_robot at
V/velocity_env_cfg.py:366-371): rl_interval_push against the oracle with injected uniforms and with the production Philox
streams, sharding, argument checks, and env.step() with the push enabled - observation rows equal to a full observation
pass after the push, everything before stage 8 unchanged, an oracle replay over several steps, the pit-terrain path and
CUDA-graph replay of the launch sequence."""
import ctypes as C

import numpy as np
import pytest
import torch

import helpers as H
import interval_events_oracle as IO
from oracle import mdp_port as port
from robot_lab_b200 import _native as nat
from robot_lab_b200.engine import MdpStepEngine
from robot_lab_b200.synthetic import MDP_KEYS, make_state
from robot_lab_b200.tasks.locomotion_velocity import push_robot_event_term

pytestmark = pytest.mark.gpu
VR = {"x": (-0.5, 0.5), "y": (-0.5, 0.5), "z": (-0.1, 0.2), "yaw": (-1.0, 1.0)}
TERM = push_robot_event_term((10.0, 15.0), VR)
SHORT = (0.01, 0.09)  # a push every 1 to 5 steps at step_dt 0.02: about an eighth of the envs fire in the first step, more later


def _bits(x: torch.Tensor) -> torch.Tensor:
    return x.detach().cpu().contiguous().view(torch.int32)


def _same_bits(a: torch.Tensor, b: torch.Tensor) -> bool:
    return torch.equal(_bits(a), _bits(b))


def _threshold_timers(n: int, dt: float, g: torch.Generator) -> torch.Tensor:
    """Timers spread over [0, 3 dt) plus, in the first envs, values whose decrement lands on and next to 1e-6."""
    t = torch.rand(n, generator=g) * 3 * dt
    edge = np.float32(np.float32(dt) + np.float32(1e-6))
    special = [np.float32(dt), np.float32(0.0), np.float32(-1.0), np.float32(15.0), edge]
    up, down = edge, edge
    for _ in range(6):
        up, down = np.nextafter(up, np.float32(1.0)), np.nextafter(down, np.float32(0.0))
        special += [up, down]
    t[:len(special)] = torch.tensor(np.array(special, dtype=np.float32))
    return t


def _kernel_setup(n: int, layout: str, seed: int):
    _, spec = H.make_spec("go2_rough")
    st = make_state(spec, n, seed=seed)
    eng = MdpStepEngine(spec, "cuda:0")
    b = eng.new_buffers(n, layout=layout)
    b.load_logical(st)
    g = torch.Generator().manual_seed(seed + 1)
    reset = torch.rand(n, generator=g) < 0.1
    term = reset & (torch.rand(n, generator=g) < 0.5)
    b.terminated.copy_(term.to(torch.uint8))
    b.truncated.copy_((reset & ~term).to(torch.uint8))
    timers = _threshold_timers(n, spec.step_dt, g)
    return spec, st, eng, b, reset, timers, g


@pytest.mark.parametrize("n,layout", [(4096, "soa"), (777, "aos"), (4096, "aos"), (777, "soa")])
def test_kernel_matches_oracle_with_injected_uniforms(native_lib, n, layout):
    spec, st, eng, b, reset, timers, g = _kernel_setup(n, layout, seed=90 + n)
    u = torch.rand(nat.RL_NUM_INTERVAL_UNIFORMS, n, generator=g)
    tl = timers.cuda()
    pushed = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    n_pushed = torch.full((1,), 12345, dtype=torch.int32, device="cuda")
    eng.interval_push(b, MdpStepEngine.interval_event_cfg(TERM), tl, pushed_ids=pushed, n_pushed=n_pushed, uniforms=u.cuda())
    torch.cuda.synchronize()
    ref = IO.interval_push(timers, st["root_lin_vel_w"], st["root_ang_vel_w"], TERM.interval_range_s, VR, spec.step_dt,
                             u, reset=reset)
    assert _same_bits(tl, ref["time_left"])
    assert _same_bits(b.logical("root_lin_vel_w"), ref["root_lin_vel_w"])
    assert _same_bits(b.logical("root_ang_vel_w"), ref["root_ang_vel_w"])
    k = int(n_pushed.item())
    ids = pushed[:k].cpu().long().sort().values
    assert torch.equal(ids, ref["pushed"].nonzero().flatten())
    assert 0 < k < n and not bool((ref["pushed"] & reset).any())   # a reset env has >= 10 s left: no push in its step
    assert bool((pushed[k:] == -1).all())
    # reset form: only the listed timers change, nothing else is touched
    ids = torch.randperm(n, generator=g)[: n // 5].to(torch.int32)
    lin0 = b.logical("root_lin_vel_w").clone()
    before = tl.cpu()
    eng.interval_push(b, MdpStepEngine.interval_event_cfg(TERM), tl, env_ids=ids.cuda(),
                      n_env_ids=torch.tensor([len(ids)], dtype=torch.int32, device="cuda"), uniforms=u.cuda())
    torch.cuda.synchronize()
    ref2 = IO.interval_push(before, st["root_lin_vel_w"], st["root_ang_vel_w"], TERM.interval_range_s, VR, spec.step_dt,
                              u, env_ids=ids)
    assert _same_bits(tl, ref2["time_left"])
    assert _same_bits(b.logical("root_lin_vel_w"), lin0)
    eng.close()


@pytest.mark.parametrize("layout", ["soa", "aos"])
def test_production_philox_draws_equal_the_oracle_streams(native_lib, layout):
    n, seed, env_off = 4096, 5, 3000
    spec, st, eng, b, reset, timers, g = _kernel_setup(n, layout, seed=17)
    cfgc = MdpStepEngine.interval_event_cfg(TERM)
    b.step_counter.fill_(4)   # device step counter 4 + step 3 = the draws of step 7
    tl = timers.cuda()
    pushed = torch.zeros(n, dtype=torch.int32, device="cuda")
    n_pushed = torch.zeros(1, dtype=torch.int32, device="cuda")
    eng.interval_push(b, cfgc, tl, pushed_ids=pushed, n_pushed=n_pushed, seed=seed, step=3, env_id_offset=env_off,
                      use_step_counter=True)
    torch.cuda.synchronize()
    u = IO.interval_uniforms(n, seed, 7, env_off)
    ref = IO.interval_push(timers, st["root_lin_vel_w"], st["root_ang_vel_w"], TERM.interval_range_s, VR, spec.step_dt,
                             u, reset=reset)
    assert _same_bits(tl, ref["time_left"])
    assert _same_bits(b.logical("root_lin_vel_w"), ref["root_lin_vel_w"])
    assert _same_bits(b.logical("root_ang_vel_w"), ref["root_ang_vel_w"])
    k = int(n_pushed.item())
    assert torch.equal(pushed[:k].cpu().long().sort().values, ref["pushed"].nonzero().flatten())
    # reset form on the Philox stream of the reset timer
    ids = torch.arange(0, n, 3, dtype=torch.int32)
    before = tl.cpu()
    eng.interval_push(b, cfgc, tl, env_ids=ids.cuda(), n_env_ids=torch.tensor([len(ids)], dtype=torch.int32, device="cuda"),
                      seed=seed, step=3, env_id_offset=env_off, use_step_counter=True)
    torch.cuda.synchronize()
    ref2 = IO.interval_push(before, st["root_lin_vel_w"], st["root_ang_vel_w"], TERM.interval_range_s, VR, spec.step_dt,
                              u, env_ids=ids)
    assert _same_bits(tl, ref2["time_left"])
    eng.close()


def test_two_shards_equal_one_launch(native_lib):
    N, cut, seed = 4096, 1536, 23
    _, spec = H.make_spec("go2_rough")
    st = make_state(spec, N, seed=seed)
    g = torch.Generator().manual_seed(seed)
    done = (torch.rand(N, generator=g) < 0.1).to(torch.uint8)
    timers = _threshold_timers(N, spec.step_dt, g)
    cfgc = MdpStepEngine.interval_event_cfg(TERM)
    eng = MdpStepEngine(spec, "cuda:0")

    def run(lo, hi):
        n = hi - lo
        b = eng.new_buffers(n)
        for k in ("root_lin_vel_w", "root_ang_vel_w"):
            b._to_device(k, st[k][lo:hi])
        b.terminated.copy_(done[lo:hi])
        b.truncated.zero_()
        tl = timers[lo:hi].clone().cuda()
        pushed = torch.zeros(n, dtype=torch.int32, device="cuda")
        n_pushed = torch.zeros(1, dtype=torch.int32, device="cuda")
        eng.interval_push(b, cfgc, tl, pushed_ids=pushed, n_pushed=n_pushed, seed=seed, step=11, env_id_offset=lo)
        torch.cuda.synchronize()
        ids = pushed[: int(n_pushed.item())].cpu().long() + lo
        return tl.cpu(), b.logical("root_lin_vel_w").cpu(), b.logical("root_ang_vel_w").cpu(), ids

    whole = run(0, N)
    a, b_ = run(0, cut), run(cut, N)
    for i in range(3):
        assert _same_bits(whole[i], torch.cat([a[i], b_[i]]))
    assert torch.equal(whole[3].sort().values, torch.cat([a[3], b_[3]]).sort().values)
    assert len(whole[3]) > 0
    eng.close()


def test_bad_arguments_are_rejected(native_lib):
    _, spec = H.make_spec("go2_rough")
    eng = MdpStepEngine(spec, "cuda:0")
    n = 64
    b = eng.new_buffers(n)
    lib, ctx = eng.lib, eng._ctx
    tl = torch.zeros(n, device="cuda")
    pushed = torch.zeros(n, dtype=torch.int32, device="cuda")
    cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
    ids = torch.arange(n, dtype=torch.int32, device="cuda")
    st = b.state_view()
    rnd = b.random()
    good = MdpStepEngine.interval_event_cfg(TERM)
    term, trunc = b.terminated.data_ptr(), b.truncated.data_ptr()

    def call(cfg=good, dt=0.02, time_left=tl.data_ptr(), state=st, terminated=term, truncated=trunc, env_ids=None,
             n_env_ids=None, pushed_ids=pushed.data_ptr(), n_pushed=cnt.data_ptr(), r=rnd):
        return lib.rl_interval_push(ctx, n, C.byref(cfg) if cfg is not None else None, dt, time_left,
                                    C.byref(state) if state is not None else None, terminated, truncated, env_ids,
                                    n_env_ids, pushed_ids, n_pushed, C.byref(r) if r is not None else None, None, 0)

    assert call() == 0
    torch.cuda.synchronize()

    def bad(**kw):
        rc = call(**kw)
        return rc == -1 and b"rl_interval_push" in lib.rl_last_error()

    assert bad(cfg=None) and bad(time_left=None) and bad(r=None)
    lohi = MdpStepEngine.interval_event_cfg(TERM)
    lohi.interval_lo, lohi.interval_hi = 3.0, 2.0
    assert bad(cfg=lohi) and b"lo <= hi" in lib.rl_last_error()
    nan = MdpStepEngine.interval_event_cfg(TERM)
    nan.interval_lo = float("nan")
    assert bad(cfg=nan)
    vel = MdpStepEngine.interval_event_cfg(TERM)
    vel.vel_lo[4], vel.vel_hi[4] = 1.0, -1.0
    assert bad(cfg=vel)
    assert bad(env_ids=ids.data_ptr())                       # env_ids without n_env_ids
    assert bad(n_env_ids=cnt.data_ptr())                     # and the other way round
    assert bad(pushed_ids=None) and bad(n_pushed=None)
    assert bad(terminated=None, truncated=None)
    assert bad(dt=0.0) and bad(dt=float("nan"))
    assert bad(state=None)
    no_vel = b.state_view(fresh=True)
    no_vel.root_ang_vel_w = nat.RlField(None, 0, 0)
    assert bad(state=no_vel)
    eng.close()


# ---- env.step() with the push enabled -------------------------------------------------------------------------------
def _env(n, phys, seed, push, pits=False):
    from robot_lab_b200.cfg import TerrainCfg
    from robot_lab_b200.envs import ManagerBasedRLEnv, ReplayStateProvider
    from robot_lab_b200.tasks import make_env_cfg

    cfg = make_env_cfg(H.TASKS["go2_rough"], num_envs=n)
    cfg.seed, cfg.sim.device = seed, "cuda:0"
    if push:
        cfg.events.randomize_push_robot = push_robot_event_term(SHORT, VR)
    if pits:
        cfg.scene.terrain = TerrainCfg(sub_terrains=("pyramid_stairs", "pits", "boxes", "random_rough", "hf_pyramid_slope"),
                                       proportions=(0.2, 0.15, 0.25, 0.3, 0.1))
    return ManagerBasedRLEnv(cfg, state_provider=ReplayStateProvider(phys))


def _reobserved(env):
    """What a full observation pass over all envs writes now (the rows are restored afterwards)."""
    b = env.buffers
    keep = [o.clone() for o in b.obs]
    env.engine.step(b, phases=nat.PHASE_OBS, **env._rng)
    torch.cuda.synchronize()
    full = [o.cpu().clone() for o in b.obs]
    for o, k in zip(b.obs, keep):
        o.copy_(k)
    return full


def test_env_step_with_push_reobserves_exactly_the_pushed_rows(native_lib):
    n, T, seed = 1024, 5, 31
    _, spec = H.make_spec("go2_rough")
    phys = [make_state(spec, n, seed=600 + t) for t in range(T + 1)]
    acts = [torch.randn(n, spec.A, generator=torch.Generator().manual_seed(t)).cuda() for t in range(T)]
    env_p, env_n = _env(n, phys, seed, True), _env(n, phys, seed, False)
    assert env_p.event_manager.available_modes == ["interval"] and env_n.event_manager.available_modes == []
    assert env_p.event_manager._interval_term_time_left[0] is env_p.interval_time_left
    assert env_p.event_manager.active_terms == {"interval": ["randomize_push_robot"]}
    env_p.reset()
    env_n.reset()
    lo, hi = SHORT
    assert bool(((env_p.interval_time_left >= lo) & (env_p.interval_time_left <= hi)).all())
    for t in range(T):
        obs_p, rew_p, term_p, trunc_p, _ = env_p.step(acts[t])
        obs_n, rew_n, term_n, trunc_n, _ = env_n.step(acts[t])
        torch.cuda.synchronize()
        k = int(env_p.n_pushed.item())
        pushed = torch.zeros(n, dtype=torch.bool)
        pushed[env_p.pushed_ids[:k].cpu().long()] = True
        assert 50 < k < n and int(pushed.sum()) == k, (t, k)
        # every row equals a full observation pass run after the push
        full = _reobserved(env_p)
        assert _same_bits(obs_p["policy"], full[0]) and _same_bits(obs_p["critic"], full[1]), t
        # everything before stage 8 is untouched by the push
        assert _same_bits(rew_p, rew_n) and torch.equal(term_p.cpu(), term_n.cpu()) and torch.equal(trunc_p.cpu(), trunc_n.cpu())
        for key in ("metric_error_vel_xy", "metric_error_vel_yaw", "command", "heading_target", "time_left",
                    "episode_sums", "episode_length"):
            assert torch.equal(env_p.buffers.logical(key).cpu(), env_n.buffers.logical(key).cpu()), (t, key)
        # only the pushed envs' rows differ
        for g in ("policy", "critic"):
            a, b = obs_p[g].cpu(), obs_n[g].cpu()
            assert _same_bits(a[~pushed], b[~pushed]), (t, g)
            assert bool((a[pushed] != b[pushed]).any(dim=1).all()), (t, g)
        assert _same_bits(env_p.buffers.logical("root_lin_vel_w")[~pushed.cuda()], env_n.buffers.logical("root_lin_vel_w")[~pushed.cuda()])
    env_p.close()
    env_n.close()


def test_env_rollout_with_push_matches_oracle_replay(native_lib):
    from robot_lab_b200.envs import ManagerBasedRLEnv, ReplayStateProvider  # noqa: F401

    n, T, seed = 768, 6, 77
    _, spec = H.make_spec("go2_rough")
    phys = [make_state(spec, n, seed=500 + t) for t in range(T)]
    actions = [torch.randn(n, spec.A, generator=torch.Generator().manual_seed(t)) for t in range(T)]
    env = _env(n, phys, seed, True)
    mdp0 = {k: phys[0][k] for k in MDP_KEYS}
    env.buffers.load_logical(mdp0)
    env.buffers.cmd_uniforms, env.buffers.obs_uniforms = None, [None, None]
    lo, hi = (torch.tensor(v, dtype=torch.float32) for v in SHORT)
    timers = IO.interval_uniforms(n, seed, 0, 0)[0] * (hi - lo) + lo       # sampled at construction (step 0)
    assert _same_bits(env.interval_time_left, timers)
    mdp = {k: v.clone() for k, v in mdp0.items()}
    keys_cmd = ("command", "heading_target", "time_left", "is_heading_env", "is_standing_env",
                "metric_error_vel_xy", "metric_error_vel_yaw")
    resets = 0
    for t in range(T):
        obs, rew, term, trunc, _ = env.step(actions[t].cuda())
        torch.cuda.synchronize()
        # oracle: ManagerBasedRLEnv.step() with stage 8 between the command update and the observations
        rnd = {"seed": seed, "step": t + 1, "env_id_offset": 0}
        action, prev, _ = port.process_action(spec, mdp, actions[t])
        mdp["action"], mdp["prev_action"] = action, prev
        out = port.step(spec, {**phys[t], **mdp}, rnd, skip_done_envs=True)
        for k in keys_cmd + ("episode_length", "episode_sums"):
            mdp[k] = out[k]
        st2, _log = port.reset_envs(spec, {**phys[t], **mdp}, out["reset_ids"], out["done_bits"], rnd)
        mdp.update(st2)
        mask = torch.zeros(n, dtype=torch.bool)
        mask[out["reset_ids"].long()] = True
        resets += int(mask.sum())
        mdp.update(port.compute_command(spec, {**phys[t], **mdp}, rnd, active=mask))
        p = IO.interval_push(timers, phys[t]["root_lin_vel_w"], phys[t]["root_ang_vel_w"], SHORT, VR, spec.step_dt,
                               IO.interval_uniforms(n, seed, t + 1, 0), reset=mask)
        timers = p["time_left"]
        ph = {**phys[t], "root_lin_vel_w": p["root_lin_vel_w"], "root_ang_vel_w": p["root_ang_vel_w"]}
        st = {**ph, **mdp}
        ref_obs = [port.compute_obs_group(spec, 0, st, rnd), port.compute_obs_group(spec, 1, st, rnd)]
        # the device side
        k = int(env.n_pushed.item())
        assert torch.equal(env.pushed_ids[:k].cpu().long().sort().values, p["pushed"].nonzero().flatten()), t
        assert _same_bits(env.interval_time_left, timers), t
        assert _same_bits(env.buffers.logical("root_lin_vel_w"), p["root_lin_vel_w"]), t
        assert _same_bits(env.buffers.logical("root_ang_vel_w"), p["root_ang_vel_w"]), t
        assert torch.equal(term.cpu(), out["terminated"]) and torch.equal(trunc.cpu(), out["truncated"]), t
        torch.testing.assert_close(rew.cpu(), out["reward"], rtol=H.RTOL, atol=H.ATOL, msg=f"step {t} reward")
        for g, name in enumerate(("policy", "critic")):
            torch.testing.assert_close(obs[name].cpu(), ref_obs[g], rtol=H.RTOL, atol=H.ATOL, msg=f"step {t} {name}")
    assert resets > 0
    env.close()


def test_env_step_on_a_terrain_with_pits_and_push(native_lib):
    n = 1024
    _, spec = H.make_spec("go2_rough")
    g = torch.Generator().manual_seed(8)
    states = []
    for i in range(4):
        st = make_state(spec, n, seed=70 + i)
        st["root_pos_w"] = torch.stack([(torch.rand(n, generator=g) - 0.5) * 70.0, (torch.rand(n, generator=g) - 0.5) * 110.0,
                                        torch.rand(n, generator=g)], dim=1)
        states.append(st)
    env = _env(n, states, 3, True, pits=True)
    assert env.pit_grid is not None
    env.reset()
    for i in range(1, 4):
        obs, _, _, _, _ = env.step(torch.zeros(n, 12, device="cuda:0"))
        torch.cuda.synchronize()
        k = int(env.n_pushed.item())
        assert k > 50
        ids = env.pushed_ids[:k].long()
        full = _reobserved(env)
        assert _same_bits(obs["policy"], full[0]) and _same_bits(obs["critic"], full[1])
        lin = env.buffers.logical("root_lin_vel_w")
        assert bool((lin[ids, :2].cpu() != states[i]["root_lin_vel_w"][ids.cpu(), :2]).any(dim=1).all())
        cmd = env.command_manager.get_command("base_velocity").cpu()
        on = env.was_on_pit.cpu().bool()
        assert ((cmd[on, 0] >= 0.3) & (cmd[on, 0] <= 0.6)).all() and (cmd[on, 1:] == 0).all()
    env.close()


def test_launch_sequence_with_push_replays_in_a_cuda_graph(native_lib):
    n, seed = 4096, 12
    _, spec = H.make_spec("go2_rough")
    eng = MdpStepEngine(spec, "cuda:0")
    b = eng.new_buffers(n)
    b.load_logical(make_state(spec, n, seed=seed))
    b.cmd_uniforms, b.obs_uniforms = None, [None, None]
    rng = dict(seed=seed, env_id_offset=0, use_random_inputs=False, use_step_counter=True)
    cfgc = MdpStepEngine.interval_event_cfg(push_robot_event_term(SHORT, VR))
    tl = torch.rand(n, generator=torch.Generator().manual_seed(1), dtype=torch.float32).cuda() * 0.1
    pushed = torch.zeros(n, dtype=torch.int32, device="cuda")
    n_pushed = torch.zeros(1, dtype=torch.int32, device="cuda")

    def one_step():
        eng.process_action(b)
        eng.step_pre_reset(b, **rng)
        eng.step_post_reset(b, **rng)
        eng.interval_push(b, cfgc, tl, pushed_ids=pushed, n_pushed=n_pushed, seed=seed, use_step_counter=True)
        eng.reobserve(b, pushed, n_pushed, **rng)

    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        one_step()                       # first calls outside capture (scratch at the full env count)
    stream.synchronize()
    state = [b.inputs.buf, b.mdp.buf, b.outputs.buf, b.done_bits, b.reset_ids, b.n_reset, b.step_counter, tl]
    snap = [x.clone() for x in state]

    def record():
        k = int(n_pushed.item())
        return {"obs0": b.obs[0].cpu().clone(), "obs1": b.obs[1].cpu().clone(), "reward": b.reward.cpu().clone(),
                "terminated": b.terminated.cpu().clone(), "truncated": b.truncated.cpu().clone(), "time_left": tl.cpu(),
                "lin": b.logical("root_lin_vel_w").cpu().clone(), "ang": b.logical("root_ang_vel_w").cpu().clone(),
                "pushed": pushed[:k].cpu().sort().values}

    eager = []
    for _ in range(3):
        with torch.cuda.stream(stream):
            one_step()
        stream.synchronize()
        eager.append(record())
    for x, s in zip(state, snap):
        x.copy_(s)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=stream):
        one_step()
    replayed = []
    for _ in range(3):
        with torch.cuda.stream(stream):
            graph.replay()
        stream.synchronize()
        replayed.append(record())
    for t, (e, r) in enumerate(zip(eager, replayed)):
        assert len(e["pushed"]) > 0, t
        for key in e:
            if e[key].dtype == torch.float32:
                assert _same_bits(e[key], r[key]), (t, key)
            else:
                assert torch.equal(e[key], r[key]), (t, key)
    eng.close()
