#!/usr/bin/env python
"""Benchmark of the per-step MDP pipeline: env-steps/s on synthetic 4096-env Unitree-Go2 rough-velocity state.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # the reference algorithm on the host CPU cores

One "step" = one pass of the hot path over one batch of synthetic env state, in the order of
ManagerBasedRLEnv.step() [IL] (SURVEY.md 3.2): process_action -> step launch 1 (terminations, rewards, reset-id
compaction) -> step launch 2 (manager reset + logging means of the done envs, command, observations). Physics /
sensors are the *producer* of the state buffers and are not part of this tier: the state is synthetic
(robot_lab_b200.synthetic) and resident in HBM before the timed region.

Timing rules followed: W >= 3 warm-up steps; the step rotates over S >= 16 independent state sets whose combined
footprint exceeds the 126 MB L2 (config.l2_policy says so); CUDA events on the launching stream with barrier +
synchronize on both sides; max over ranks; nvidia-smi clocks sampled during the timed region. The K timed steps are
ONE OR TWO CUDA-graph launches whatever K is (whole 24-step rollouts + one remainder graph captured during warm-up).
Prints ONE JSON line on rank 0.

Keys beside the contract's: roofline (dominant kernel at the headline size), roofline_large_n (the same two kernels
at 65536 envs, where bytes - not launch latency - decide), e2e (host buffers through the C-ABI, with the PCIe ceiling of
the same box measured beside it and the Python API step timed), cpu_baseline, handoff / value_incl_handoff /
shard_parity (N > 1), l2_resident, neighbours.
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

TASK_DEFAULT = "RobotLab-Isaac-Velocity-Rough-Unitree-Go2-v0"
METRIC = "env-steps/sec (4096-env Go2 rough-velocity)"
UNIT = "env-steps/s"
ROLLOUT = 24  # steps per PPO rollout (GO2/agents/rsl_rl_ppo_cfg.py:11) = steps per captured CUDA graph
NVLINK_PEER_GBS = 770.0   # measured peer-copy bandwidth per direction per GPU on this pool (B200_PROFILING.md)


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=2400)
    p.add_argument("--warmup", type=int, default=240)
    p.add_argument("--impl", choices=["ours", "reference"], default="ours")
    p.add_argument("--task", default=TASK_DEFAULT)
    p.add_argument("--num-envs", type=int, default=4096, help="envs per GPU (weak scaling)")
    p.add_argument("--sets", type=int, default=24, help="independent state sets the step rotates over (L2 defeat)")
    p.add_argument("--warps", type=int, default=0, help="general kernel: warps per tile (4/8/16; a tile is 32 envs)")
    p.add_argument("--pdl", choices=["on", "off"], default="off",
                   help="programmatic dependent launch between the kernels of a step (measured: no gain, profiles/r2_summary.md)")
    p.add_argument("--no-graph", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the bounded CPU baseline sample")
    p.add_argument("--skip-handoff", action="store_true")
    p.add_argument("--no-verify", action="store_true", help="N > 1: skip the sharded-vs-single-GPU parity check")
    p.add_argument("--large-n", type=int, default=65536, help="env count of roofline_large_n (0 = skip)")
    p.add_argument("--no-neighbours", action="store_true", help="skip the side measurements of the SURVEY 8(f) kernels")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write what the last timed step returned to its caller as DIR/<name>.npy (rank 0)")
    return p.parse_args()


def workload_string(task: str, n: int) -> str:
    """The SAME string in both arms (the driver compares the two lines' config)."""
    tag = " (BASELINE.json configs[2])" if task == TASK_DEFAULT and n == 4096 else ""
    return f"{task}{tag}, {n} envs/GPU, full MDP step (process_action + terminations/rewards/reset ids + manager reset/command/observations)"


# ---------------------------------------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md "clocks DURING the timed region")
# ---------------------------------------------------------------------------------------------------------
class ClockSampler:
    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [x.strip() for x in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for nm, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        # "under load" = the samples taken while the GPU was clocked up (an idle GPU parks at ~120 MHz)
        busy = [x for x in sm if x > 0.5 * max(mx)] if mx else []
        return {"sm_mhz": statistics.median(busy) if busy else (statistics.median(sm) if sm else None),
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm),
                "samples_under_load": len(busy)}


# ---------------------------------------------------------------------------------------------------------
# CPU reference arm / cpu_baseline: the oracle port (eager fp32 torch, the reference's own op stream) on host cores
# ---------------------------------------------------------------------------------------------------------
def cpu_step_fn(spec, st):
    from oracle import mdp_port as port

    rnd = {"cmd_uniforms": st["cmd_uniforms"], "obs_uniforms_policy": st["obs_uniforms_policy"],
           "obs_uniforms_critic": st["obs_uniforms_critic"]}

    def one_step():
        action, prev, _target = port.process_action(spec, st, st["new_action"])
        s1 = dict(st)
        s1["action"], s1["prev_action"] = action, prev
        out = port.step(spec, s1, rnd, skip_done_envs=True)
        s2 = dict(s1)
        s2.update({k: out[k] for k in ("command", "heading_target", "time_left", "is_heading_env", "is_standing_env",
                                       "metric_error_vel_xy", "metric_error_vel_yaw", "episode_length", "episode_sums")})
        s3, _log = port.reset_envs(spec, s2, out["reset_ids"], out["done_bits"], rnd)
        s2.update(s3)
        mask = torch.zeros(st["root_quat_w"].shape[0], dtype=torch.bool)
        mask[out["reset_ids"].long()] = True
        s2.update(port.compute_command(spec, s2, rnd, active=mask))
        port.compute_obs_group(spec, 0, s2, rnd)
        port.compute_obs_group(spec, 1, s2, rnd)
        return out["reward"]

    return one_step


def time_cpu(spec, num_envs: int, steps: int, warmup: int, budget_s: float | None):
    from robot_lab_b200.synthetic import make_state

    st = make_state(spec, num_envs)
    fn = cpu_step_fn(spec, st)
    # eager torch on [4096, C] tensors is dispatch-bound: more intra-op threads can be slower. Give the CPU arm
    # its best case: sweep the thread count (2 steps each) and keep the fastest.
    ncpu = os.cpu_count() or 1
    sweep, best = {}, None
    for nt in sorted({1, 2, 4, 8, 16, 32, 64, ncpu}):
        if nt > ncpu:
            continue
        torch.set_num_threads(nt)
        fn()
        t0 = time.perf_counter()
        fn()
        sweep[nt] = time.perf_counter() - t0
        if best is None or sweep[nt] < sweep[best]:
            best = nt
    cores = best
    torch.set_num_threads(cores)
    for _ in range(max(1, warmup)):
        fn()
    t0 = time.perf_counter()
    done = 0
    while done < steps:
        fn()
        done += 1
        if budget_s is not None and time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return {"value": num_envs * done / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{done} full MDP steps of {num_envs} envs ({dt:.1f} s), eager fp32 torch oracle port, "
                      f"torch.set_num_threads({cores}) = fastest of a sweep over {sorted(sweep)} threads on {ncpu} logical CPUs",
            "ms_per_step": 1e3 * dt / done, "steps": done}


def run_reference(args, spec, rank: int, world: int):
    """--impl reference: the reference's CPU implementation of the path (oracle port; the reference's own
    Python files cannot travel to the GPU box) on this box's host cores. Rank 0 only. Same steps / warm-up / config
    keys as the GPU arm; a step is one full MDP step of num_envs envs (~18 ms), so even the default K ends in a minute
    (a 150 s budget bounds absurd K; the line then reports the steps actually taken)."""
    if rank != 0:
        return
    W = max(3, args.warmup)
    res = time_cpu(spec, args.num_envs, args.steps, min(W, 10), budget_s=150.0)
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps if res["steps"] == args.steps else res["steps"], "warmup": W, "ms_per_step": res["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_string(args.task, args.num_envs), "num_envs_per_gpu": args.num_envs},
        "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "warm-up steps beyond 10 are not run on the CPU arm (each costs ~18 ms and changes nothing); the timed "
                "steps are full-size MDP steps",
    }
    _emit(line)


# ---------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------
_JSON_OUT = None   # the process's real stdout, kept for the ONE JSON line


def _emit(line: dict) -> None:
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    global _JSON_OUT
    args = parse_args()
    # stdout carries exactly one JSON line. Libraries write there too (NCCL prints its version banner to fd 1 whatever
    # NCCL_DEBUG_FILE says): keep a private copy of fd 1 for the JSON line and point fd 1 at stderr for everything else.
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    from robot_lab_b200.spec import compact_layout, compile_step_spec
    from robot_lab_b200.tasks import make_env_cfg

    cfg = make_env_cfg(args.task, num_envs=args.num_envs)
    spec = compile_step_spec(cfg, compact_layout(cfg))

    if args.impl == "reference":
        run_reference(args, spec, rank, world)
        return

    import torch.distributed as dist

    from robot_lab_b200.engine import MdpStepEngine
    from robot_lab_b200.synthetic import make_state

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the MDP step has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL's version banner / debug lines go to stdout by default: keep stdout to the ONE JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)

    N, S, K, W = args.num_envs, max(1, args.sets), args.steps, max(3, args.warmup)
    eng = MdpStepEngine(spec, dev)
    if args.warps:
        eng.set_launch_config(args.warps, 0)
    use_pdl = args.pdl == "on"
    eng.set_pdl(use_pdl)

    # ---- N > 1: sharded-vs-single-GPU parity, before anything is timed ----
    shard_parity = None
    if world > 1 and not args.no_verify:
        shard_parity = verify_shards(spec, N, rank, world, dev, local_rank)

    sets = []
    for i in range(S):
        b = eng.new_buffers(N)
        b.load_logical(make_state(spec, N, seed=1234 + 1000 * i, rank=rank))
        b.cmd_uniforms, b.obs_uniforms = None, [None, None]  # production mode: in-kernel Philox, no noise bytes
        sets.append(b)
    env_off = rank * N
    rng = dict(seed=42 + rank, env_id_offset=env_off, use_random_inputs=False, use_step_counter=True)

    def one_step(b):
        # ManagerBasedRLEnv.step() [IL]: process_action -> (physics: the synthetic provider changes nothing) ->
        # terminations, rewards, reset ids -> (external reset) -> manager reset, command, observations
        eng.process_action(b)
        eng.step_pre_reset(b, **rng)
        eng.step_post_reset(b, **rng)

    launches_per_step = 3
    stream = torch.cuda.Stream(device=dev)
    # ---- untimed: first calls (scratch allocation, tensor maps), then graph capture ----
    with torch.cuda.stream(stream):
        for b in sets:
            one_step(b)
    stream.synchronize()

    def capture(n_steps: int, first_set: int = 0):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=stream):
            for i in range(n_steps):
                one_step(sets[(first_set + i) % S])
        return g

    use_graph = not args.no_graph
    G = ROLLOUT
    graphs: dict[int, torch.cuda.CUDAGraph] = {}

    def graph_of(n_steps: int):
        if n_steps not in graphs:
            graphs[n_steps] = capture(n_steps)
            # one untimed replay: the first launch of an instantiated graph also uploads it to the device (~0.1 ms), which
            # must not land in a timed region that replays this graph only once (K < 24, e.g. the driver's --steps 20)
            with torch.cuda.stream(stream):
                graphs[n_steps].replay()
            stream.synchronize()
        return graphs[n_steps]

    def run_steps(n: int) -> None:
        """Exactly n steps on `stream`: whole rollouts replay the 24-step graph, the remainder ONE graph of n % 24 steps
        (both captured before the timed region) - the timed K steps are at most two kinds of graph launches."""
        with torch.cuda.stream(stream):
            if not use_graph:
                for i in range(n):
                    one_step(sets[i % S])
                return
            q, r = divmod(n, G)
            for _ in range(q):
                graphs[G].replay()
            if r:
                graphs[r].replay()

    if use_graph:
        for n_ in {G, K % G, W % G} - {0}:
            graph_of(n_)
    run_steps(W)           # warm-up (>= 3 steps)
    stream.synchronize()
    # the clock-sampler spin-up below runs a time-dependent number of steps: on a state set of its own, so that the timed
    # steps start from the state the warm-up left and the same arguments give them the same inputs
    spin = None
    if use_graph:
        spare = eng.new_buffers(N)
        spare.load_logical(make_state(spec, N, seed=1234 + 1000 * S, rank=rank))
        spare.cmd_uniforms, spare.obs_uniforms = None, [None, None]
        with torch.cuda.stream(stream):
            one_step(spare)
        stream.synchronize()
        spin = torch.cuda.CUDAGraph()
        with torch.cuda.graph(spin, stream=stream):
            for _ in range(G):
                one_step(spare)

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize(dev)

    # ---- timed region: exactly K steps ----
    sampler = ClockSampler(local_rank)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    if rank == 0:
        sampler.start()
    # 0.25 s for the clock sampler to spin up - with the GPU under load (untimed replays of the rollout graph), not idle:
    # an idle quarter second lets the GPU drop its clocks, and a short timed region (the driver's --steps 20 is 0.45 ms)
    # would be measured on the ramp. Then the barrier + synchronize the contract asks for, and the timed region at once.
    t_keep0 = time.perf_counter()
    while time.perf_counter() - t_keep0 < 0.25:
        if use_graph:
            with torch.cuda.stream(stream):
                for _ in range(20):
                    spin.replay()
            stream.synchronize()
        else:
            time.sleep(0.05)
    barrier()
    t_wall0 = time.perf_counter()
    ev0.record(stream)
    run_steps(K)
    ev1.record(stream)
    stream.synchronize()
    barrier()
    t_wall = time.perf_counter() - t_wall0
    elapsed_ms = ev0.elapsed_time(ev1)
    last_outputs = None
    if args.dump_outputs and rank == 0:   # read now: everything after the timed region steps the same sets again
        last_set = ((K - 1) % G if use_graph else K - 1) % S
        last_outputs = step_outputs(spec, sets[last_set])
    if rank == 0 and t_wall < 1.0 and use_graph:
        # nvidia-smi samples every 100 ms: keep the same graphs running (untimed) long enough for the clock record to
        # show the GPU under load
        t_keep = time.perf_counter()
        while time.perf_counter() - t_keep < 1.0:
            with torch.cuda.stream(stream):
                for _ in range(50):
                    graphs[G].replay()
            stream.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    if world > 1:
        barrier()
        tmax = torch.tensor([elapsed_ms], device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        elapsed_ms = float(tmax.item())
    value = world * N * K / (elapsed_ms * 1e-3)
    ms_per_step = elapsed_ms / K

    # ---- each step kernel alone for the roofline: same rotation, graph of G back-to-back launches ----
    def time_kernel(fn, set_list=None, reps_cap=200):
        ss = set_list if set_list is not None else sets
        with torch.cuda.stream(stream):
            for b in ss:
                fn(b)
        stream.synchronize()
        gk = torch.cuda.CUDAGraph()
        n_l = max(G, len(ss)) if set_list is None else 2 * len(ss)
        with torch.cuda.graph(gk, stream=stream):
            for i in range(n_l):
                fn(ss[i % len(ss)])
        reps = max(3, min(reps_cap, K // G))
        with torch.cuda.stream(stream):
            for _ in range(3):
                gk.replay()
            k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            k0.record(stream)
            for _ in range(reps):
                gk.replay()
            k1.record(stream)
        stream.synchronize()
        return 1e3 * k0.elapsed_time(k1) / (reps * n_l)

    peaks_path = ROOT / "MEASURED_PEAKS.json"
    if peaks_path.exists():
        peak, peak_src = float(json.loads(peaks_path.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"
    traffic_db = {}
    tp = ROOT / "profiles" / "traffic_latest.json"
    if tp.exists():
        try:
            traffic_db = json.loads(tp.read_text())
        except Exception:
            traffic_db = {}

    def kernel_name(e, n, kind):
        cc = e.cluster_config(n)
        if cc["cluster_size"] == 0:
            return f"mdp_step_kernel ({'DONES|REWARDS|COMPACT' if kind == 'pre_reset' else 'RESET|COMMAND|OBS'}, general kernel)"
        which = "v2_pre_kernel (DONES|REWARDS|COMPACT)" if kind == "pre_reset" else "v2_post_kernel (RESET|COMMAND|OBS)"
        return f"{which}, cluster {cc['cluster_size']} x {cc['tiles_per_cta']} tiles x {cc['warps_per_cta']} warps"

    def roofline_of(e, set_list, n, step_us=None, reps_cap=200, with_traffic=False):
        e_rng = dict(rng)
        kernels = {}
        for kind, fn in (("pre_reset", lambda b: e.step_pre_reset(b, **e_rng)), ("post_reset", lambda b: e.step_post_reset(b, **e_rng))):
            us = time_kernel(fn, set_list, reps_cap)
            nbytes = spec.algorithmic_bytes_per_launch(kind) * n
            achieved = nbytes / (us * 1e-6) / 1e9
            tr = traffic_db.get(kind, {}) if with_traffic else {}
            kernels[kind] = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": tr.get("dram_bytes_per_launch"),
                             "traffic_source": (f"ncu --set full, {tr.get('captured', 'capture date unknown')}, kernel "
                                                f"{tr.get('kernel', '?')}: a stored capture, not a measurement of this run")
                             if tr.get("dram_bytes_per_launch") is not None else None,
                             "kernel": kernel_name(e, n, kind), "kernel_us": us, "bytes_per_launch": nbytes,
                             "bytes_per_env": spec.algorithmic_bytes_per_launch(kind), "peak_source": peak_src}
            if step_us:
                kernels[kind]["kernel_share_of_step"] = us / step_us
        dom = max(kernels, key=lambda k: kernels[k]["kernel_us"])
        out = dict(kernels[dom])
        out["other_kernel"] = kernels["post_reset" if dom == "pre_reset" else "pre_reset"]
        return out

    roofline = roofline_of(eng, None, N, step_us=ms_per_step * 1e3, with_traffic=(N == 4096 and args.task == TASK_DEFAULT))
    roofline["bytes_per_env_step_fused_accounting"] = spec.algorithmic_bytes_per_env_step()
    roofline["whole_step"] = {"achieved": spec.algorithmic_bytes_per_env_step() * N / (ms_per_step * 1e-3) / 1e9,
                              "frac": spec.algorithmic_bytes_per_env_step() * N / (ms_per_step * 1e-3) / 1e9 / peak,
                              "note": "SURVEY 8(d) bytes per env-step x N / ms_per_step (three launches)"}

    # ---- the same kernels where bytes - not launch latency - decide: 65536 envs (16 waves of tiles) ----
    roofline_large_n = None
    if rank == 0 and args.large_n and args.large_n != N:
        roofline_large_n = measure_large_n(spec, args.large_n, dev, rng, roofline_of, stream)

    # ---- the neighbours of the path (SURVEY.md 8(f)): each kernel alone, same rotation over the state sets ----
    neighbours = None
    if rank == 0 and world == 1 and not args.no_neighbours:
        neighbours = measure_neighbours(eng, spec, sets, N, time_kernel, peak, dev)

    # ---- the same step with an L2-resident working set (one state set, 14 MB): labelled separately (SURVEY 8(d)) ----
    l2_resident = None
    if use_graph and not args.no_e2e:
        g1 = torch.cuda.CUDAGraph()
        with torch.cuda.stream(stream):
            for _ in range(3):
                one_step(sets[0])
        stream.synchronize()
        with torch.cuda.graph(g1, stream=stream):
            for _ in range(G):
                one_step(sets[0])
        with torch.cuda.stream(stream):
            for _ in range(3):
                g1.replay()
            r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps1 = max(3, min(100, K // G))
            r0.record(stream)
            for _ in range(reps1):
                g1.replay()
            r1.record(stream)
        stream.synchronize()
        ms1 = r0.elapsed_time(r1) / (reps1 * G)
        l2_resident = {"value": world * N * 1e3 / ms1, "unit": UNIT, "ms_per_step": ms1,
                       "note": "single state set (working set < L2); the headline value rotates over sets larger than L2"}

    # ---- e2e: same step through the C-ABI with HOST buffers (pinned), H2D + D2H inside the timed region ----
    e2e = None
    if not args.no_e2e:
        e2e = measure_e2e(eng, spec, sets, N, K, W, rank, world, dev, local_rank, one_step)
        if rank == 0 and world == 1:
            e2e["api"] = measure_api_step(args.task, N, dev)

    # ---- multi-GPU hand-off (the one exchange of the path: rollout all-gather at the PPO boundary) ----
    handoff, value_incl_handoff = None, None
    if world > 1 and not args.skip_handoff:
        handoff = measure_handoff(eng, spec, sets, N, world, dev, local_rank, one_step)
        value_incl_handoff = handoff.pop("value_incl_handoff")

    # ---- CPU baseline (rank 0, N=1 run only) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        res = time_cpu(spec, N, steps=10_000, warmup=2, budget_s=args.cpu_seconds)
        cpu = {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {
                "workload": workload_string(args.task, N), "num_envs_per_gpu": N,
                "shape": f"J={spec.J} B={spec.B} F={spec.Bt} R={spec.R} K={spec.K}, policy/critic rows {spec.obs[0].dim}/{spec.obs[1].dim}",
                "state_sets": S, "cuda_graph_steps": G if use_graph else 0,
                "timed_region": ((f"{K // G} x {G}-step graph" + (f" + 1 x {K % G}-step graph" if K % G else "")) if use_graph else "eager launches"),
                "pdl": use_pdl, "launch": eng.cluster_config(N) | {"general_kernel": eng.launch_config()},
                "l2_policy": f"rotating over {S} independent state sets (inputs+outputs+manager state "
                             f"{S * (sets[0].inputs.nbytes + sets[0].outputs.nbytes + sets[0].mdp.nbytes) / 1e6:.0f} MB > 126 MB L2)",
                "noise": "in-kernel Philox4x32-10 (0 bytes)", "parallelism": f"dp{world} (env shards, no data-path collective)",
            },
            "gpu_launches": launches_per_step * K,
            "clocks": clocks, "roofline": roofline, "roofline_large_n": roofline_large_n, "e2e": e2e, "cpu_baseline": cpu,
            "handoff": handoff, "value_incl_handoff": value_incl_handoff, "shard_parity": shard_parity,
            "l2_resident": l2_resident, "neighbours": neighbours,
            "wall_s_timed_region": t_wall,
        }
        _emit(line)
    if last_outputs is not None:
        write_outputs(Path(args.dump_outputs), last_outputs)
    if world > 1:
        dist.destroy_process_group()


DUMP_LIMIT_BYTES = 64 * 10**6 - 4096   # 64 MB in all, .npy headers included


def step_outputs(spec, b) -> tuple[dict, dict]:
    """What the caller of one env step receives, copied to the host: per-env arrays (observation rows of each group,
    reward, done masks, the joint targets of the processed action) and the others (reset ids, reset logging means)."""
    per_env = {f"obs_{grp.name}": b.obs[g] for g, grp in enumerate(spec.obs) if b.obs[g] is not None}
    per_env.update(reward=b.reward, terminated=b.terminated, truncated=b.truncated, joint_target=b.logical("joint_target"))
    per_env = {k: v.float().cpu() for k, v in per_env.items()}
    other = {"reset_ids": b.reset_ids[: int(b.n_reset.item())].double().cpu(), "reset_log": b.log_all.float().cpu()}
    return per_env, other


def write_outputs(out_dir: Path, outputs: tuple[dict, dict]) -> None:
    """One float32 / float64 .npy file per array. Beyond 64 MB in all, the per-env arrays keep a fixed, seeded sample of
    env rows, listed in env_ids.npy."""
    import numpy as np

    per_env, other = outputs
    n = next(iter(per_env.values())).shape[0]
    nbytes = sum(v.numel() * v.element_size() for v in per_env.values())
    budget = DUMP_LIMIT_BYTES - sum(v.numel() * v.element_size() for v in other.values()) - 8 * n
    if nbytes > budget:
        keep = n * budget // nbytes
        ids = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:keep].sort().values
        per_env = {k: v[ids] for k, v in per_env.items()}
        other = {**other, "env_ids": ids.double()}
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, v in {**per_env, **other}.items():
        np.save(out_dir / f"{name}.npy", v.contiguous().numpy())


def measure_large_n(spec, n_large, dev, rng, roofline_of, stream):
    """The two step kernels at n_large envs (default 65536 = 2048 tiles, ~14 waves): the regime where the HBM roofline -
    not launch latency - is the bound. Two state sets (each ~0.4 GB of inputs + results: far beyond L2)."""
    from robot_lab_b200.engine import MdpStepEngine
    from robot_lab_b200.synthetic import make_state

    eng = MdpStepEngine(spec, dev)
    eng.set_pdl(False)
    try:
        ss = []
        for i in range(2):
            b = eng.new_buffers(n_large)
            b.load_logical(make_state(spec, n_large, seed=777 + i))
            b.cmd_uniforms, b.obs_uniforms = None, [None, None]
            ss.append(b)
        with torch.cuda.stream(stream):
            for b in ss:
                eng.process_action(b)
        out = roofline_of(eng, ss, n_large, reps_cap=20)
        us_pa = None
        g = torch.cuda.CUDAGraph()
        with torch.cuda.stream(stream):
            for b in ss:
                eng.process_action(b); eng.step_pre_reset(b, **rng); eng.step_post_reset(b, **rng)
        stream.synchronize()
        with torch.cuda.graph(g, stream=stream):
            for _ in range(4):
                for b in ss:
                    eng.process_action(b); eng.step_pre_reset(b, **rng); eng.step_post_reset(b, **rng)
        with torch.cuda.stream(stream):
            g.replay()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(5):
                g.replay()
            e1.record(stream)
        stream.synchronize()
        us_step = 1e3 * e0.elapsed_time(e1) / (5 * 8)
        out["num_envs"] = n_large
        out["env_step_us"] = us_step
        out["env_steps_per_s"] = n_large / (us_step * 1e-6)
        out["whole_step_frac"] = spec.algorithmic_bytes_per_env_step() * n_large / (us_step * 1e-6) / 1e9 / out["peak"]
        out["note"] = ("same kernels, same accounting as `roofline`, one GPU, 2 state sets rotating (each beyond L2); "
                       "frac = the slower of the two step kernels, other_kernel beside it")
        return out
    finally:
        eng.close()


def measure_neighbours(eng, spec, sets, N, time_kernel, peak, dev):
    """Side measurements (not part of `value`): the SURVEY.md 8(f) kernels that run around the step in a simulator
    loop - per physics sub-step the actuator model and the contact-sensor update, per env step the height scanner, per
    env step on pit terrains the command restriction. bytes = per-env tensors read + written (the height field and the
    terrain origins are shared, L2-resident tables)."""
    from robot_lab_b200 import terrain as terrain_host
    from robot_lab_b200.cfg import RayCasterCfg, TerrainCfg

    out = {}

    def add(name, fn, bytes_per_env, note):
        us = time_kernel(fn)
        gbs = bytes_per_env * N / (us * 1e-6) / 1e9
        out[name] = {"kernel_us": us, "bytes_per_env": bytes_per_env, "achieved_gbs": gbs, "frac_of_hbm_peak": gbs / peak,
                     "note": note}

    J, R, B, Bt, T = spec.J, spec.R, spec.B, spec.Bt, spec.T
    add("rl_process_action", lambda b: eng.process_action(b), 4 * 5 * spec.A,
        "reads the policy's action rows + the stored action, writes previous / stored action and the joint targets")
    add("rl_actuator_step", lambda b: eng.actuator_step(b), 4 * 4 * J,
        "DCMotor: reads target, joint_pos, joint_vel, writes applied_torque; x decimation per env step")
    forces = torch.randn(N, B, 3, device=dev)
    add("rl_contact_sensor_update(ring)", lambda b: eng.contact_sensor_update(b, forces, 0.005, ring_slot=1),
        4 * (3 * B + 3 * B + 6 * Bt), "reads net_forces_w, writes one history slot, read-modify-writes 4 timers")
    if R > 0:
        ter = TerrainCfg()
        nx = int(round((ter.num_rows * ter.size[0] + 2 * ter.border_width) / ter.horizontal_scale)) + 1
        ny = int(round((ter.num_cols * ter.size[1] + 2 * ter.border_width) / ter.horizontal_scale)) + 1
        g = torch.Generator(device="cpu").manual_seed(7)
        heights = (torch.rand(nx // 8 + 2, ny // 8 + 2, generator=g) * 0.8)
        heights = torch.nn.functional.interpolate(heights[None, None], size=(nx, ny), mode="bilinear", align_corners=True)[0, 0]
        hf = terrain_host.HeightFieldBuffers(heights.contiguous().to(dev), -0.5 * (nx - 1) * ter.horizontal_scale,
                                             -0.5 * (ny - 1) * ter.horizontal_scale, ter.horizontal_scale,
                                             terrain_host.grid_pattern_ray_starts(RayCasterCfg()).to(dev))
        add("rl_height_scan_cast", lambda b: eng.height_scan_cast(b, hf), 4 * (7 + R + 1),
            f"{R} vertical rays per env over a {nx} x {ny} height field ({nx * ny * 4 / 1e6:.1f} MB, L2-resident gathers)")
    pit = TerrainCfg(sub_terrains=("pyramid_stairs", "pits", "boxes", "random_rough", "hf_pyramid_slope"),
                     proportions=(0.2, 0.15, 0.25, 0.3, 0.1))
    grid = terrain_host.TerrainGridBuffers.create(pit, "pits", dev)
    was = torch.zeros(N, dtype=torch.uint8, device=dev)
    add("rl_command_pit_restrict", lambda b: eng.command_pit_restrict(b, grid, was, seed=1, use_random_inputs=False),
        4 * 2 + 2, "argmin over 200 terrain origins per env (shared memory) + command rewrite for pit envs")
    return out


def _numa_pin(dev, local_rank):
    """Restrict this process to the CPUs next to the GPU while pinned staging buffers are first touched (a remote NUMA
    node costs up to 40 % of the PCIe rate on a two-socket host). Returns (description, restore-callable)."""
    old_aff = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    try:
        props = torch.cuda.get_device_properties(dev)
        if all(hasattr(props, k) for k in ("pci_domain_id", "pci_bus_id", "pci_device_id")):
            bdf = f"{int(props.pci_domain_id):04x}:{int(props.pci_bus_id):02x}:{int(props.pci_device_id):02x}.0"
        else:
            import pynvml
            pynvml.nvmlInit()
            bdf = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(dev.index if dev.index is not None else local_rank)).busId
            bdf = (bdf.decode() if isinstance(bdf, bytes) else bdf).lower()
            if len(bdf.split(":")[0]) == 8:
                bdf = bdf[4:]
        cpus = Path(f"/sys/bus/pci/devices/{bdf}/local_cpulist").read_text().strip()
        want = set()
        for part in cpus.split(","):
            lo, _, hi = part.partition("-")
            want.update(range(int(lo), int(hi or lo) + 1))
        want &= old_aff
        if want:
            os.sched_setaffinity(0, want)
            desc = f"pinned buffers first-touched on the CPUs local to GPU {bdf} ({cpus})"
        else:
            desc = f"GPU {bdf}: local CPUs {cpus} not in this process's affinity mask"
    except Exception as e:   # not fatal: the buffers land wherever the allocator puts them
        desc = f"no NUMA placement ({type(e).__name__})"

    def restore():
        if old_aff is not None:
            try:
                os.sched_setaffinity(0, old_aff)
            except Exception:
                pass

    return desc, restore


def measure_e2e(eng, spec, sets, N, K, W, rank, world, dev, local_rank, one_step):
    """Every step: one H2D copy of that step's inputs (physics/sensor state + policy action) from pinned host
    memory, the three launches, one D2H read of the step's results (observation rows, reward, done masks).
    Three streams pipeline copy-in / compute / copy-out over a ring of device sets. The PCIe ceiling of the box is
    measured in the same call: the same two copies, same sizes, same streams, no kernels."""
    import torch.distributed as dist

    ring = min(4, len(sets))
    dsets = sets[:ring]
    in_bytes, out_bytes = dsets[0].inputs.nbytes, dsets[0].outputs.nbytes
    numa, restore = _numa_pin(dev, local_rank)
    host_in = [torch.empty(in_bytes, dtype=torch.uint8).pin_memory() for _ in range(ring)]
    host_out = [torch.empty(out_bytes, dtype=torch.uint8).pin_memory() for _ in range(ring)]
    for h, b in zip(host_in, dsets):
        h.copy_(b.inputs.buf[:in_bytes].cpu())
    for h in host_out:
        h.zero_()
    restore()
    s_in, s_cmp, s_out = (torch.cuda.Stream(device=dev) for _ in range(3))
    ev_in = [torch.cuda.Event() for _ in range(ring)]
    ev_cmp = [torch.cuda.Event() for _ in range(ring)]
    ev_out = [torch.cuda.Event() for _ in range(ring)]
    steps = max(200, min(K, 600))   # its own step count: long enough for the 4-deep pipeline to reach steady state

    # the three launches of a set, captured once through the C-ABI calls: replaying them keeps the host side of a
    # step at a handful of stream operations (the Python / ctypes cost of three rl_* calls would otherwise bound it)
    graphs = []
    with torch.cuda.stream(s_cmp):
        for b in dsets:
            one_step(b)
    torch.cuda.synchronize(dev)
    for b in dsets:
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s_cmp):
            one_step(b)
        graphs.append(g)

    def run(n, with_compute=True):
        for i in range(n):
            r = i % ring
            b = dsets[r]
            with torch.cuda.stream(s_in):
                s_in.wait_event(ev_cmp[r])          # the set's previous compute has consumed its inputs
                b.inputs.buf[:in_bytes].copy_(host_in[r], non_blocking=True)
                ev_in[r].record(s_in)
            with torch.cuda.stream(s_cmp):
                s_cmp.wait_event(ev_in[r])
                s_cmp.wait_event(ev_out[r])         # the set's previous results have been read back
                if with_compute:
                    graphs[r].replay()
                ev_cmp[r].record(s_cmp)
            with torch.cuda.stream(s_out):
                s_out.wait_event(ev_cmp[r])
                host_out[r].copy_(b.outputs.buf[:out_bytes], non_blocking=True)
                ev_out[r].record(s_out)

    def timed(n, with_compute):
        run(max(24, min(W, 48)), with_compute)
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier(device_ids=[local_rank])
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(s_in)
        run(n, with_compute)
        for s in (s_in, s_cmp):
            s_out.wait_stream(s)
        t1.record(s_out)
        torch.cuda.synchronize(dev)
        ms = t0.elapsed_time(t1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    ms_copy = timed(steps, with_compute=False)     # the ceiling: the same copies, nothing in between
    ms = timed(steps, with_compute=True)
    ms_copy = min(ms_copy, timed(steps, with_compute=False))   # ... taken before and after (the first pass also warms the path)
    h2d, d2h = dsets[0].input_bytes(), dsets[0].output_bytes()
    ceiling = world * N * steps / (ms_copy * 1e-3)
    return {"value": world * N * steps / (ms * 1e-3), "unit": UNIT,
            "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
            "steps": steps, "ms_per_step": ms / steps, "numa": numa,
            "pcie": {"copies_only_ms_per_step": ms_copy / steps, "ceiling_env_steps_per_s": ceiling,
                     "h2d_gbs": h2d / (ms_copy / steps * 1e-3) / 1e9, "d2h_gbs": d2h / (ms_copy / steps * 1e-3) / 1e9,
                     "note": "the same pinned H2D + D2H copies per step on the same streams with NO kernels in between: what "
                             "this box's PCIe path delivers for these sizes (both directions concurrently)"},
            "frac_of_pcie": (ms_copy / ms),
            "path": "pinned host buffers -> 1 H2D -> rl_process_action + 2 x rl_step (C-ABI calls captured once, replayed as a CUDA graph) -> 1 D2H per step, 3-stream pipeline over a ring of 4 device sets"}


def measure_api_step(task, N, dev):
    """The call rsl_rl makes: RslRlVecEnvWrapper.step(actions) - eager Python, three C-ABI launches, a state provider
    whose state is already resident (the producer is not part of this tier), results returned as device tensors. Wall
    clock per call with the device kept busy (the calls are asynchronous: this is the HOST cost of a step, the bound of
    an eager training loop), and the device time per call."""
    from robot_lab_b200 import envs
    from robot_lab_b200.tasks import make_env_cfg

    cfg = make_env_cfg(task, num_envs=N)
    cfg.sim.device = str(dev)

    class Resident(envs.StateProvider):
        def advance(self, env):
            return

    env = envs.RslRlVecEnvWrapper(envs.ManagerBasedRLEnv(cfg, state_provider=Resident()))
    from robot_lab_b200.synthetic import make_state

    env.unwrapped.buffers.load_logical(make_state(env.unwrapped.spec, N, seed=5))
    env.unwrapped.buffers.cmd_uniforms, env.unwrapped.buffers.obs_uniforms = None, [None, None]
    actions = torch.randn(N, env.num_actions, device=dev)
    for _ in range(50):
        env.step(actions)
    torch.cuda.synchronize(dev)
    n = 1000
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(n):
        env.step(actions)
    e1.record()
    t_host = time.perf_counter() - t0
    torch.cuda.synchronize(dev)
    dev_us = 1e3 * e0.elapsed_time(e1) / n
    out = {"api_step_us": 1e6 * t_host / n, "api_step_device_us": dev_us, "env_steps_per_s": N * n / max(t_host, e0.elapsed_time(e1) * 1e-3),
           "call": "RslRlVecEnvWrapper.step(actions): eager Python -> rl_process_action + 2 x rl_step through ctypes, resident state"}
    env.close()
    return out


def verify_shards(spec, N, rank, world, dev, local_rank):
    """configs[4] on hardware: every rank steps its shard (env_id_offset = rank * N, the production Philox streams, two
    env steps); the results are gathered and rank 0 compares them with ONE single-GPU run over all world * N envs:
    masks and reset ids bit-exact, floats to 1e-5 (they come out bit-identical: same kernels, same counters)."""
    import torch.distributed as dist

    from robot_lab_b200.engine import MdpStepEngine
    from robot_lab_b200.synthetic import make_state

    total = world * N
    steps = 2
    states = [make_state(spec, total, seed=4242 + t) for t in range(steps)]   # the same global state on every rank

    def run(eng, n, lo, offset):
        b = eng.new_buffers(n)
        outs = []
        for t, st in enumerate(states):
            part = {k: (v[:, lo:lo + n] if k == "cmd_uniforms" else v[lo:lo + n]) for k, v in st.items()}
            if t > 0:   # fresh physics + action; the manager state chains
                part = {k: v for k, v in part.items() if k in _STATE_KEYS or k == "new_action"}
            b.load_logical(part)
            b.cmd_uniforms, b.obs_uniforms = None, [None, None]
            kw = dict(seed=99, env_id_offset=offset, use_random_inputs=False, use_step_counter=True)
            eng.process_action(b)
            eng.step_pre_reset(b, **kw)
            eng.step_post_reset(b, **kw)
            torch.cuda.synchronize(dev)
            done = (b.terminated | b.truncated)
            outs.append({"obs0": b.obs[0].clone(), "obs1": b.obs[1].clone(), "reward": b.reward.clone(),
                         "terminated": b.terminated.clone(), "truncated": b.truncated.clone(), "done": done.clone(),
                         "n_reset": int(b.n_reset.item()), "reset_ids": b.reset_ids[: int(b.n_reset.item())].clone() + offset,
                         "command": b.logical("command").contiguous().clone(), "sums": b.logical("episode_sums").contiguous().clone(),
                         "eplen": b.logical("episode_length").clone()})
        return outs

    from robot_lab_b200 import _native as nat
    _STATE_KEYS = set(nat._STATE_FIELDS)
    eng = MdpStepEngine(spec, dev)
    mine = run(eng, N, rank * N, rank * N)
    eng.close()
    report = {"ok": True, "envs": total, "steps": steps, "max_abs_float_diff": 0.0, "compared": []}
    keys_f = ("obs0", "obs1", "reward", "command", "sums")
    keys_x = ("terminated", "truncated", "eplen")
    gathered = []
    for t in range(steps):
        g = {}
        for k in keys_f + keys_x:
            x = mine[t][k].contiguous()
            outl = [torch.empty_like(x) for _ in range(world)]
            dist.all_gather(outl, x)
            g[k] = torch.cat(outl, dim=0)
        cnt = torch.tensor([mine[t]["n_reset"]], device=dev)
        cl = [torch.zeros_like(cnt) for _ in range(world)]
        dist.all_gather(cl, cnt)
        ids = torch.full((N,), -1, dtype=torch.int32, device=dev)
        ids[: mine[t]["n_reset"]] = mine[t]["reset_ids"]
        il = [torch.empty_like(ids) for _ in range(world)]
        dist.all_gather(il, ids)
        g["reset_ids"] = torch.cat([il[r][: int(cl[r].item())] for r in range(world)])
        gathered.append(g)
    if rank == 0:
        eng1 = MdpStepEngine(spec, dev)
        ref = run(eng1, total, 0, 0)
        eng1.close()
        for t in range(steps):
            for k in keys_x + ("reset_ids",):
                same = gathered[t][k].shape == ref[t][k].shape and torch.equal(gathered[t][k], ref[t][k])
                report["ok"] = report["ok"] and bool(same)
                report["compared"].append(f"step{t}.{k}:{'exact' if same else 'MISMATCH'}")
            for k in keys_f:
                a, b_ = gathered[t][k].float(), ref[t][k].float()
                fin = torch.isfinite(a) & torch.isfinite(b_)
                d = float((a[fin] - b_[fin]).abs().max()) if fin.any() else 0.0
                okk = bool(torch.allclose(a, b_, rtol=1e-5, atol=1e-6, equal_nan=True))
                report["ok"] = report["ok"] and okk
                report["max_abs_float_diff"] = max(report["max_abs_float_diff"], d)
                report["compared"].append(f"step{t}.{k}:{'bit-identical' if torch.equal(a, b_) else ('within 1e-5' if okk else 'MISMATCH')}")
        report["resets_per_step"] = [int(gathered[t]["reset_ids"].numel()) for t in range(steps)]
    dist.barrier(device_ids=[local_rank])
    return report if rank == 0 else None


def measure_handoff(eng, spec, sets, N, world, dev, local_rank, one_step):
    """The one exchange of the path (north_star: "NCCL over NVLink only at the rollout-buffer all-gather hand-off to PPO";
    reference recipe README.md:323-337, train.py:143-150). One rollout = 24 env steps; every rank needs every rank's slab.

      compute_only   the 24 steps alone (one CUDA graph), results written in place into the rollout slabs
      unstreamed     the same, then ONE all-gather of the whole rollout
      streamed       per-step graphs; the all-gather of a chunk of slabs is issued on a side stream the moment its last step is
                     done and runs while the next steps compute (RolloutStorage.gather_step; chunk sizes 1, 2, 4, 8 are all
                     measured, the best one is the headline); the clock stops when the last gather lands
      floor          (world - 1) * steps * N * width * 4 bytes must enter every GPU through its own NVLink ingress

    value_incl_handoff = world * N * 24 / streamed time. Also: rsl_rl's own multi-GPU mode (gradient all-reduce instead
    of a rollout gather) for scale."""
    import torch.distributed as dist

    from robot_lab_b200.rollout import RolloutStorage

    S = len(sets)
    store = RolloutStorage(spec, N, ROLLOUT, dev)
    main = torch.cuda.Stream(device=dev)
    # the step launches of set t write their results into slab t (no copy into the rollout)
    for t in range(ROLLOUT):
        store.bind(sets[t % S], t)
    with torch.cuda.stream(main):
        for t in range(ROLLOUT):
            one_step(sets[t % S])
    main.synchronize()
    g_all = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g_all, stream=main):
        for t in range(ROLLOUT):
            one_step(sets[t % S])
    g_step = []
    for t in range(ROLLOUT):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=main):
            one_step(sets[t % S])
        g_step.append(g)

    def timed(fn, reps=10):
        for _ in range(2):
            fn()
        torch.cuda.synchronize(dev)
        dist.barrier(device_ids=[local_rank])
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(main):
            e0.record(main)
            for _ in range(reps):
                fn()
            e1.record(main)
        torch.cuda.synchronize(dev)
        t = torch.tensor([e0.elapsed_time(e1) / reps], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def compute_only():
        with torch.cuda.stream(main):
            g_all.replay()

    def unstreamed():
        with torch.cuda.stream(main):
            g_all.replay()
            store.gather_all()

    def streamed():
        with torch.cuda.stream(main):
            for t in range(ROLLOUT):
                g_step[t].replay()
                store.gather_step(t, after=main)
            store.finish()

    def gather_only():
        with torch.cuda.stream(main):
            store.gather_all()

    ms_c, ms_u, ms_g = timed(compute_only), timed(unstreamed), timed(gather_only)
    # chunking of the streamed gather: launch latency of a collective against how early it can start
    sweep = {}
    for k in (1, 2, 4, 8):
        store.set_gather_every(k)
        sweep[k] = timed(streamed)
    best_k = min(sweep, key=sweep.get)
    store.set_gather_every(best_k)
    ms_s = sweep[best_k]
    # the whole streamed rollout - 24 steps on the main stream, the chunk gathers forked onto the side stream, the join - as
    # ONE CUDA graph (NCCL collectives are capturable): no host work between the steps at all
    ms_sg, graph_note = None, None
    try:
        torch.cuda.synchronize(dev)
        dist.barrier(device_ids=[local_rank])
        g_stream = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g_stream, stream=main):
            for t in range(ROLLOUT):
                one_step(sets[t % S])
                store.gather_step(t, after=main)
            store.finish()

        def streamed_graph():
            with torch.cuda.stream(main):
                g_stream.replay()

        ms_sg = timed(streamed_graph)
        if ms_sg < ms_s:
            ms_s, graph_note = ms_sg, "whole streamed rollout (steps + side-stream gathers) replayed as one CUDA graph"
    except Exception as e:   # capture of collectives not supported in this build: keep the eager pipeline's number
        graph_note = f"graph capture of the streamed rollout failed ({type(e).__name__}): eager pipeline timed"
        torch.cuda.synchronize(dev)
    nbytes = store.data.numel() * 4
    ingress = nbytes * (world - 1)
    floor_ms = ingress / (NVLINK_PEER_GBS * 1e9) * 1e3
    # rsl_rl's own multi-GPU hand-off: 20 gradient all-reduces (5 epochs x 4 mini-batches) of the actor-critic's flat
    # gradient (512-256-128 MLPs on 45 / 235 inputs: ~0.48 M parameters = 1.9 MB) per iteration
    n_param = sum(a * b + b for a, b in ((spec.obs[0].dim, 512), (512, 256), (256, 128), (128, spec.A),
                                         (spec.obs[1].dim, 512), (512, 256), (256, 128), (128, 1))) + spec.A
    grad = torch.randn(n_param, device=dev)
    def grad_allreduce():
        with torch.cuda.stream(main):
            for _ in range(20):
                dist.all_reduce(grad)
    ms_gr = timed(grad_allreduce, reps=5)
    for b in sets:   # give the state sets their own outputs back
        b.rebind_outputs(obs=[b.outputs.views[f"obs{g}"] if grp.dim > 0 else None for g, grp in enumerate(spec.obs)],
                         reward=b.outputs.views["reward"], terminated=b.outputs.views["terminated"], truncated=b.outputs.views["truncated"])
    return {"collective": "ncclAllGather per env step on a side stream (torch.distributed over NVLink 5 / NVSwitch), results written "
                          "in place into per-step rollout slabs",
            "bytes_per_rank_per_rollout": nbytes, "ingress_bytes_per_rank": ingress, "per_rollout_steps": ROLLOUT,
            "compute_only_ms": ms_c, "unstreamed_ms": ms_u, "streamed_ms": ms_s, "gather_alone_ms": ms_g,
            "streamed_ms_by_steps_per_gather": sweep, "steps_per_gather": best_k, "streamed_graph_ms": ms_sg, "streamed_note": graph_note,
            "exposed_handoff_ms": ms_s - ms_c, "exposed_handoff_ms_unstreamed": ms_u - ms_c,
            "floor_ms": floor_ms, "floor_note": f"{ingress / 1e6:.0f} MB must enter every GPU; {NVLINK_PEER_GBS:.0f} GB/s measured peer copy per "
                                                "direction per GPU (900 nominal): NVLink INGRESS per GPU is the limiting link",
            "bus_gbs_streamed": ingress / (ms_s * 1e-3) / 1e9, "bus_gbs_gather_alone": ingress / (ms_g * 1e-3) / 1e9,
            "efficiency_vs_compute_only": ms_c / ms_s,
            "gradient_allreduce_alternative": {"ms_per_iteration": ms_gr, "bytes_per_allreduce": n_param * 4, "allreduces": 20,
                                               "note": "rsl_rl's own multi-GPU mode keeps rollouts local and all-reduces gradients "
                                                       "(SURVEY.md section 5); it overlaps with the backward pass of the learner, which "
                                                       "is outside this tier"},
            "value_incl_handoff": world * N * ROLLOUT / (ms_s * 1e-3)}


if __name__ == "__main__":
    main()
