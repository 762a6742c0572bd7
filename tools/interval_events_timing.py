"""Cost of the interval push event (rl_interval_push, stage 8 of the env step) on the GPU, at 4096 and 65536 envs.

Usage (GPU box): python tools/interval_events_timing.py [--out profiles/interval_events_timing.json] [--task go2_rough]

Measured, each over state sets whose total footprint is larger than the 126 MB L2 (sets are rotated, so every launch
reads state that no earlier launch of the window left in L2), with CUDA events around replays of captured CUDA graphs:
  * ``push_alone``: rl_interval_push (memset of the count + the step kernel) alone, per launch;
  * ``step_base``: the env step without the push - process_action, DONES|REWARDS|COMPACT, RESET|COMMAND|OBS (fused);
  * ``step_fused_push``: the same + rl_interval_push + rl_step(OBS) over the pushed ids (what env.step() runs);
  * ``step_split_push``: process_action, DONES|REWARDS|COMPACT, RESET|COMMAND, rl_interval_push, OBS over all envs.
The term is the reference's (10 to 15 s, +-0.5 m/s in x / y) at step_dt 0.02 s, timers spread over [0, 15) s as in a running
env: about one env in 600 is pushed per step.
The card's name and power limit are read in the same run and written next to the numbers.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

import torch  # noqa: E402

import helpers as H  # noqa: E402
from robot_lab_b200 import _native as nat  # noqa: E402
from robot_lab_b200.engine import MdpStepEngine  # noqa: E402
from robot_lab_b200.synthetic import make_state  # noqa: E402
from robot_lab_b200.tasks.locomotion_velocity import push_robot_event_term  # noqa: E402

L2_BYTES = 126 * 2**20


def card() -> dict:
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
    except Exception as e:  # pragma: no cover - reported, not hidden
        out = f"nvidia-smi unavailable: {e}"
    return {"torch_device_name": torch.cuda.get_device_name(0), "nvidia_smi": out}


def time_graph(fn, stream, launches: int, reps: int) -> dict:
    """us per `launches` unit of fn() captured once; fn() enqueues exactly one such unit per call."""
    with torch.cuda.stream(stream):
        fn()
    stream.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=stream):
        fn()
    with torch.cuda.stream(stream):
        g.replay()   # upload
    stream.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    samples = []
    for _ in range(3):
        with torch.cuda.stream(stream):
            e0.record(stream)
            for _ in range(reps):
                g.replay()
            e1.record(stream)
        stream.synchronize()
        samples.append(e0.elapsed_time(e1) * 1e3 / (reps * launches))
    return {"us": min(samples), "samples_us": samples}


def run(n: int, task: str) -> dict:
    _, spec = H.make_spec(task)
    eng = MdpStepEngine(spec, "cuda:0")
    term = push_robot_event_term()
    cfgc = MdpStepEngine.interval_event_cfg(term)
    rng = dict(seed=42, env_id_offset=0, use_random_inputs=False, use_step_counter=True)
    prng = dict(seed=42, use_step_counter=True)
    stream = torch.cuda.Stream()
    lo, hi = term.interval_range_s

    # ---- env step variants: rotating StateBuffers sets --------------------------------------------------------------
    probe = eng.new_buffers(n)
    per_set = probe.inputs.nbytes + probe.mdp.nbytes + probe.outputs.nbytes
    S = max(4, -(-2 * L2_BYTES // per_set))
    sets = [probe]
    for i in range(S - 1):
        sets.append(eng.new_buffers(n))
    ev = []
    for i, b in enumerate(sets):
        b.load_logical(make_state(spec, n, seed=1234 + 1000 * i))
        b.cmd_uniforms, b.obs_uniforms = None, [None, None]
        # timers spread over [0, hi): the steady state of a running env, in which about dt / 12.5 s of the envs fire per step
        ev.append({"tl": torch.rand(n, device="cuda") * hi, "ids": torch.zeros(n, dtype=torch.int32, device="cuda"),
                   "n": torch.zeros(1, dtype=torch.int32, device="cuda")})

    def push(i):
        b, e = sets[i], ev[i]
        eng.interval_push(b, cfgc, e["tl"], pushed_ids=e["ids"], n_pushed=e["n"], **prng)

    def step_base(i):
        b = sets[i]
        eng.process_action(b)
        eng.step_pre_reset(b, **rng)
        eng.step_post_reset(b, **rng)

    def step_fused_push(i):
        step_base(i)
        push(i)
        eng.reobserve(sets[i], ev[i]["ids"], ev[i]["n"], **rng)

    def step_split_push(i):
        b = sets[i]
        eng.process_action(b)
        eng.step_pre_reset(b, **rng)
        eng.step(b, phases=nat.PHASE_RESET | nat.PHASE_COMMAND, **rng)
        push(i)
        eng.step(b, phases=nat.PHASE_OBS, **rng)

    res = {"num_envs": n, "task": task, "env_sets": S, "env_set_bytes": per_set, "env_sets_total_mb": S * per_set / 2**20}
    with torch.cuda.stream(stream):
        for i in range(S):
            step_fused_push(i)
            step_split_push(i)
    stream.synchronize()
    reps = max(2, 2000 // S) if n <= 8192 else max(2, 400 // S)
    for name, fn in (("step_base", step_base), ("step_fused_push", step_fused_push), ("step_split_push", step_split_push),
                     ("step_base_again", step_base)):
        res[name] = time_graph(lambda fn=fn: [fn(i) for i in range(S)], stream, S, reps)
    with torch.cuda.stream(stream):
        step_fused_push(0)
    stream.synchronize()
    res["pushed_per_step_sample"] = int(ev[0]["n"].item())

    # ---- rl_interval_push alone: its own state (timers, root velocities, done bytes, id list) rotated over > L2 ------
    per_env = 4 + 6 * 4 + 2 + 4
    M = max(4, -(-2 * L2_BYTES // (per_env * n)))
    tl = torch.rand(M, n, device="cuda") * hi
    vel = torch.randn(M, 2, 3, n, device="cuda")
    done = (torch.rand(M, 2, n, device="cuda") < 0.005).to(torch.uint8)
    ids = torch.zeros(M, n, dtype=torch.int32, device="cuda")
    cnt = torch.zeros(M, dtype=torch.int32, device="cuda")
    rnd = probe.random(42, 0, 0, False, True)
    views = []
    for m in range(M):
        st = nat.RlStateView()
        st.root_lin_vel_w = nat.field_of(vel[m, 0], "soa")
        st.root_ang_vel_w = nat.field_of(vel[m, 1], "soa")
        views.append(st)
    lib, ctx = eng.lib, eng._ctx

    def alone():
        s = torch.cuda.current_stream().cuda_stream
        for m in range(M):
            nat.check(lib.rl_interval_push(ctx, n, C.byref(cfgc), float(spec.step_dt), tl[m].data_ptr(), C.byref(views[m]),
                                           done[m, 0].data_ptr(), done[m, 1].data_ptr(), None, None, ids[m].data_ptr(),
                                           cnt[m:m + 1].data_ptr(), C.byref(rnd), None, s))

    res["push_alone"] = time_graph(alone, stream, M, max(2, 4000 // M))
    res.update({"push_sets": M, "push_sets_total_mb": M * per_env * n / 2**20})
    res["push_cost_fused_us"] = res["step_fused_push"]["us"] - res["step_base"]["us"]
    res["push_cost_split_us"] = res["step_split_push"]["us"] - res["step_base"]["us"]
    eng.close()
    return res


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--out", default=str(ROOT / "profiles" / "interval_events_timing.json"))
    p.add_argument("--task", default="go2_rough")
    p.add_argument("--envs", default="4096,65536")
    args = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("interval_events_timing.py measures on a CUDA device; there is nothing to measure without one")
    out = {"card": card(), "results": [run(int(n), args.task) for n in args.envs.split(",")]}
    out["card_after"] = card()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1) + "\n")
    for r in out["results"]:
        print(f"N={r['num_envs']}: push alone {r['push_alone']['us']:.2f} us; step base {r['step_base']['us']:.2f} / "
              f"again {r['step_base_again']['us']:.2f}, fused+push+reobserve {r['step_fused_push']['us']:.2f}, "
              f"split {r['step_split_push']['us']:.2f} us per env step; pushed/step ~{r['pushed_per_step_sample']}")
    print(json.dumps(out["card"]))


if __name__ == "__main__":
    main()
