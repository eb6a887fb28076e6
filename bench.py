#!/usr/bin/env python
"""Benchmark of the fused CollectiveCrossing step kernel (contract: see the task statement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (config.workload): BASELINE.json configs[1] geometry and policy — the README 12x8 grid
with 5 boarding + 3 exiting agents, DefaultReward, IndividualAtDestination, MaxSteps 100, greedy
baseline policy evaluated inside the step kernel, auto-reset — at 1,048,576 envs per GPU (the
north_star's roofline size; the per-step working set of 1.4 GB is far larger than L2, so no
flush is needed between iterations).  A "step" is one fused kernel launch over all envs.
Metric: agent-steps/s = env-steps x 8 agent slots, whole job.
"""

from __future__ import annotations

import argparse
import json
import os
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
for p in (str(ROOT), str(ROOT / "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = "agent_steps_per_sec"
UNIT = "agent-steps/s"
DUMP_BYTES = 48 * 10**6   # --dump-outputs: at most this many bytes of .npy data


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=1 << 20, help="envs per GPU")
    ap.add_argument("--obs-dtype", default="float32", choices=["float32", "int8", "none"])
    ap.add_argument("--policy", default="greedy", choices=["greedy", "waiting", "random"])
    ap.add_argument("--steps-per-launch", type=int, default=20,
                    help="env-steps fused into one launch (cc_rollout_fused); 1 = one launch per step")
    ap.add_argument("--reps", type=int, default=5, help="repetitions of the timed region (the median is reported)")
    ap.add_argument("--e2e-steps", type=int, default=24)
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary measurements")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step (obs, reward, agent_flags, env_flags, actions) as DIR/<name>.npy "
                         "in float32; above %d MB a fixed, seeded sample of envs (rank 0's shard with --gpus > 1)" % (DUMP_BYTES // 10**6))
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    return args


def workload_config():
    from cases import readme_config

    return readme_config()


def config_dict(args, n_total):
    return {
        "workload": f"BASELINE configs[1]: README 12x8 grid, door 5-7, 5 boarding + 3 exiting agents, DefaultReward, "
                    f"IndividualAtDestination, MaxSteps 100, {args.policy} baseline policy in-kernel, auto-reset; "
                    f"{args.envs} envs per GPU",
        "envs_total": n_total, "envs_per_gpu": args.envs, "agents_per_env": 8, "obs_dtype": args.obs_dtype,
        "policy": args.policy, "steps_per_launch_max": args.steps_per_launch,
        "launch": (f"cc_rollout_fused: up to {args.steps_per_launch} env-steps per launch (see roofline.steps_per_launch), state in registers, "
                   f"every step's outputs written ([T, N, ...] buffers); steps % T as single-step launches"
                   if args.steps_per_launch > 1 else "cc_step: one launch per env-step"),
        "l2_policy": "inputs larger than L2 (no flush)" if args.envs >= 1 << 19 else "working set may fit L2",
        "episode_phases": "step counters spread uniformly over [0, MaxSteps) after reset(): every step sees the steady-state share of episode ends",
        "parallelism": "independent env shards, one process per GPU, no data-path collective",
    }


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled through NVML every few milliseconds on a host thread (the
    timed region lasts tens of milliseconds, far less than one `nvidia-smi -lms` period).  Only
    the samples taken between mark_begin() and mark_end() — the timed region — are summarised."""

    BAD = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}
    NOTED = {"sw_power_cap": 0x4}

    def __init__(self, gpu_index: int, period_s: float = 0.002):
        import threading

        self.rows, self.t_begin, self.t_end, self.err = [], None, None, None
        self._stop = threading.Event()
        try:
            import pynvml

            pynvml.nvmlInit()
            # NVML enumerates physical devices: honour CUDA_VISIBLE_DEVICES when it holds plain indices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            ids = [v for v in vis.split(",") if v.strip().isdigit()]
            phys = int(ids[gpu_index]) if gpu_index < len(ids) else gpu_index
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as exc:  # noqa: BLE001 - no NVML, no clocks
            self.err, self.thread = f"NVML unavailable: {exc}", None
            return
        self.period = period_s
        self.thread = threading.Thread(target=self._run, daemon=True)
        self.thread.start()

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                try:
                    power = nv.nvmlDeviceGetPowerUsage(self.h) / 1e3
                except Exception:  # noqa: BLE001
                    power = float("nan")
                self.rows.append((time.perf_counter(), float(mhz), int(reasons), power))
            except Exception as exc:  # noqa: BLE001
                self.err = str(exc)
                return
            self._stop.wait(self.period)

    def mark_begin(self):
        self.t_begin = time.perf_counter()

    def mark_end(self):
        self.t_end = time.perf_counter()

    def stop(self) -> dict:
        if self.thread is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [self.err]}
        self._stop.set()
        self.thread.join(timeout=2)
        t0, t1 = self.t_begin or 0.0, self.t_end or float("inf")
        rows = [r for r in self.rows if t0 <= r[0] <= t1]
        if not rows:   # region shorter than one sample period: the nearest samples on either side
            rows = sorted(self.rows, key=lambda r: min(abs(r[0] - t0), abs(r[0] - t1)))[:2]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [self.err or "no samples"]}
        sm = sorted(r[1] for r in rows)
        seen = 0
        for r in rows:
            seen |= r[2]
        reasons = [nm for nm, bit in {**self.BAD, **self.NOTED}.items() if seen & bit]
        return {"sm_mhz": sm[len(sm) // 2], "sm_min_mhz": sm[0], "sm_max_mhz": self.max_mhz, "samples": len(rows),
                "power_w_max": max(r[3] for r in rows), "reasons": reasons, "source": "NVML, samples inside the timed region"}


# ------------------------------------------------------------------------------------------------
# CPU legs (the only places bench.py touches oracle/)
# ------------------------------------------------------------------------------------------------
def cpu_c_oracle(args, seconds):
    """The C oracle (OpenMP, all host threads) on a bounded sample of the same workload."""
    import oracle
    from collectivecrossing_b200 import _abi
    from collectivecrossing_b200.lowering import lower_config

    cores = os.cpu_count() or 1
    n = 65536
    code = {"float32": _abi.OBS_FP32, "int8": _abi.OBS_INT8, "none": _abi.OBS_NONE}[args.obs_dtype]
    orc = oracle.OracleEnvs(lower_config(workload_config()), n, seed=1)
    orc.reset()
    for _ in range(2):
        orc.step(policy=args.policy, auto_reset=True, obs_dtype=code)
    t0 = time.perf_counter()
    steps = 0
    while time.perf_counter() - t0 < seconds and steps < 400:
        orc.step(policy=args.policy, auto_reset=True, obs_dtype=code)
        steps += 1
    dt = time.perf_counter() - t0
    return {"value": n * 8 * steps / dt, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"C oracle (oracle/cc_oracle.c, OpenMP x{cores}): {n} envs x {steps} steps of the same workload in {dt:.1f} s"}


def _py_worker(job):
    policy, seconds, seed = job
    from oracle.pyport import PyEnv

    env = PyEnv(workload_config())
    env.reset(seed=seed)
    for _ in range(50):
        env.step(env.policy_actions(policy) if policy != "random" else {})
    t0 = time.perf_counter()
    steps = 0
    import numpy as np
    rng = np.random.default_rng(seed)
    while time.perf_counter() - t0 < seconds:
        for _ in range(100):
            acts = env.policy_actions(policy) if policy != "random" else {i: int(rng.integers(0, 5)) for i in env.agents}
            _, _, term, trunc, _ = env.step(acts)
            steps += 1
            if term["__all__"] or trunc["__all__"]:
                env.reset()
    return steps, time.perf_counter() - t0


_REF_STATE = {}


def _ref_worker(job):
    """The UNMODIFIED reference (oracle/refload.py: /root/reference or the staged archive): its CollectiveCrossingEnv.step
    (collectivecrossing.py:161-261) driven by its own GreedyPolicy / WaitingPolicy at epsilon 0 in the loop of
    scripts/run_greedy_policy_demo.py:67-109, reset() on episode end."""
    policy, seconds, seed = job
    import logging

    import numpy as np

    logging.disable(logging.CRITICAL)   # the reference's policies log every construction
    st = _REF_STATE
    if "env" not in st:
        from oracle import refload

        ref = refload.load()
        st["env"] = ref.CollectiveCrossingEnv(refload.to_reference_config(workload_config()))
        st["policies"] = {"greedy": ref.GreedyPolicy(0.0, 42), "waiting": ref.WaitingPolicy(0.0, 42)}
        st["obs"], _ = st["env"].reset(seed=seed)
        st["term"] = {}
    env, pol = st["env"], st["policies"].get(policy)
    rng = np.random.default_rng(seed)
    obs, terminateds = st["obs"], st["term"]
    t0 = time.perf_counter()
    steps = 0
    while time.perf_counter() - t0 < seconds:
        for _ in range(20):
            actions = {}
            for agent_id in env.agents:                                   # run_greedy_policy_demo.py:71-77
                if agent_id in obs and not terminateds.get(agent_id, False) and env._agents[agent_id].active:
                    actions[agent_id] = pol.get_action(agent_id, obs[agent_id], env) if pol else int(rng.integers(0, 5))
            obs, _, terminateds, truncateds, _ = env.step(actions)
            steps += 1
            if terminateds["__all__"] or truncateds["__all__"]:
                obs, _ = env.reset()
                terminateds = {}
    st["obs"], st["term"] = obs, terminateds
    return steps, time.perf_counter() - t0


def reference_available() -> bool:
    try:
        from oracle import refload

        return refload.available()
    except Exception:  # noqa: BLE001
        return False


def cpu_python_loop(args, seconds, pool=None):
    """The reference's own shape of computation: a pure-Python env + policy loop, one independent env per host core
    (multiprocessing), reset() on episode end (BASELINE.md §3).  The unmodified reference itself where it is available
    (kind "reference"), else the oracle's Python port of the same loop (kind "port")."""
    import multiprocessing as mp

    cores = os.cpu_count() or 1
    own = pool is None
    if own:
        pool = mp.get_context("spawn").Pool(cores)
    real = reference_available()
    try:
        res = pool.map(_ref_worker if real else _py_worker, [(args.policy, seconds, 1000 + k) for k in range(cores)])
    finally:
        if own:
            pool.close()
    rate = sum(s / dt for s, dt in res) * 8
    what = ("the unmodified reference (CollectiveCrossingEnv.step + its own baseline policy at epsilon 0, loop of "
            "scripts/run_greedy_policy_demo.py:67-109; imported from the archive oracle/stage_ref.py stages)" if real
            else "pure-Python port of the reference loop (oracle/pyport.py)")
    return {"value": rate, "unit": UNIT, "cores": cores, "kind": "reference" if real else "port",
            "sample": f"{what}, {cores} processes x 1 env, {sum(s for s, _ in res)} env-steps in {seconds:.1f} s each, "
                      f"{args.policy} policy + step + reset on done"}


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path on all host cores — the unmodified reference
    where oracle/_ref holds its archive (or /root/reference is mounted), else the oracle's Python port.  A step is a bounded
    sample: every core runs the loop for a fixed time slice."""
    import multiprocessing as mp

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    total = args.warmup + args.steps
    slice_s = max(0.25, min(4.0, 100.0 / max(1, total)))
    vals, info = [], None
    with mp.get_context("spawn").Pool(os.cpu_count() or 1) as pool:
        for k in range(total):
            info = cpu_python_loop(args, slice_s, pool)
            if k >= args.warmup:
                vals.append(info["value"])
    value = sum(vals) / len(vals)
    info["value"] = value
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": len(vals),
        "warmup": args.warmup, "ms_per_step": slice_s * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "python int / float64", "data": "synthetic", "config": config_dict(args, args.envs * args.gpus),
        "cpu_baseline": info, "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def time_steps(env, torch, dist, args, steps, policy, world, per_launch=1, sharded=None):
    """ONE timed region: EXACTLY `steps` env-steps of every env — steps // per_launch fused launches of `per_launch` steps
    (all of whose observations, rewards and flags are written) and steps % per_launch single-step launches — bracketed by
    barrier + synchronize, CUDA events on the launching stream, max over ranks.  With `sharded` (world > 1) the episode
    statistics are all-reduced (NCCL) once per launch INSIDE the region, enqueued behind the kernels with no host wait.
    Returns (ms, reduced statistics tensor or None)."""
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stats_t = None
    e0.record()
    if per_launch > 1:
        for _ in range(steps // per_launch):
            env.rollout_trajectory(per_launch, policy=policy)
            if sharded is not None:
                stats_t = sharded.global_stats_device()
        steps = steps % per_launch
    for _ in range(steps):
        env.step(policy=policy)
        if sharded is not None:
            stats_t = sharded.global_stats_device()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=env.device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
        dist.barrier()
    return ms, stats_t


def desynchronise(env, torch):
    """After reset() every env is at step 0, so all of them would hit MaxSteps in the same step, every 100 steps.  Spread the
    episode phases (step counters uniform in [0, max_steps)): every step then sees the steady-state share of finished episodes."""
    hi = int(env.cfg.max_steps)
    if hi > 1:
        g = torch.Generator(device=env.device)
        g.manual_seed(1234 + env.global_env_offset)
        env.step_count.copy_(torch.randint(0, hi, (env.num_envs,), generator=g, device=env.device, dtype=torch.int32))


def dump_outputs(out_dir, outputs, torch):
    """Write the step outputs in `outputs` (name -> device tensor with the env index first, or None) as out_dir/<name>.npy in
    float32.  Where they exceed DUMP_BYTES, the same envs of every output are kept: a sorted sample drawn with a fixed seed, so
    that two builds run with the same arguments can be compared file for file."""
    import numpy as np

    outputs = {k: v for k, v in outputs.items() if v is not None}
    n = next(iter(outputs.values())).shape[0]
    per_env = sum(4 * v[0].numel() for v in outputs.values())
    keep = min(n, DUMP_BYTES // per_env)
    idx = None
    if keep < n:
        idx = torch.from_numpy(np.sort(np.random.default_rng(0).choice(n, keep, replace=False))).to(next(iter(outputs.values())).device)
    os.makedirs(out_dir, exist_ok=True)
    for name, v in outputs.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), (v if idx is None else v.index_select(0, idx)).float().cpu().numpy())
    print(f"dumped the last timed step's outputs of {keep} of {n} envs to {out_dir}", file=sys.stderr)


def median(vals):
    v = sorted(vals)
    return v[len(v) // 2] if len(v) % 2 else 0.5 * (v[len(v) // 2 - 1] + v[len(v) // 2])


def bind_to_gpu_numa_node(gpu_index: int):
    """Run this rank on the CPU cores NVML reports as local to its GPU, so that the pinned host buffers of the
    host-buffer path are first-touched on the GPU's NUMA node (8 ranks x 1.3 GB per step otherwise cross sockets)."""
    try:
        import pynvml

        pynvml.nvmlInit()
        vis = [v for v in os.environ.get("CUDA_VISIBLE_DEVICES", "").split(",") if v.strip().isdigit()]
        phys = int(vis[gpu_index]) if gpu_index < len(vis) else gpu_index
        h = pynvml.nvmlDeviceGetHandleByIndex(phys)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (word >> b) & 1 and 64 * w + b < n_cpu}
        allowed = os.sched_getaffinity(0)
        if cpus & allowed:
            os.sched_setaffinity(0, cpus & allowed)
        return allowed   # restored before the CPU baseline runs on all host threads
    except Exception:  # noqa: BLE001 - no NVML / no affinity support: run unbound
        return None


def host_copy_bandwidth(torch):
    """Host-memory copy bandwidth with every host thread (torch CPU copy of 1 GiB): context for the host-buffer path."""
    try:
        a = torch.ones(1 << 28, dtype=torch.float32)
        b = torch.empty_like(a)
        b.copy_(a)
        t0 = time.perf_counter()
        for _ in range(3):
            b.copy_(a)
        return 3 * 2 * a.numel() * 4 / (time.perf_counter() - t0) / 1e9
    except Exception:  # noqa: BLE001
        return None


def time_e2e(env, torch, dist, world, policy, steps, host, T=1, on_device_policy=False):
    """The host-buffer path a numpy / RLlib caller binds, timed by wall clock AND CUDA events (the larger counts), max over
    ranks: per step the actions come from HOST memory (pinned) and every output lands in HOST memory (cc_step_host); with
    T > 1 one cc_rollout_host call rolls T steps out with the on-device policy.  Returns ms per env-step."""
    n, A = env.num_envs, env.num_agents
    dev_actions = torch.zeros((n, A), dtype=torch.int8, device=env.device)

    def one():
        if T > 1:
            env.rollout_host(host, T, policy=policy)
        elif on_device_policy:
            env.step_host(host, policy=policy)
        else:
            env.policy_actions(policy, out=dev_actions)            # stands in for the caller's host-side policy ...
            host["actions"].copy_(dev_actions, non_blocking=True)  # ... whose actions are in host memory
            torch.cuda.current_stream().synchronize()
            env.step_host(host)

    for _ in range(2):
        one()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t0 = time.perf_counter()
    calls = max(1, steps // T)
    for _ in range(calls):
        one()
    wall = (time.perf_counter() - t0) * 1e3
    e1.record()
    torch.cuda.synchronize()
    ms = max(e0.elapsed_time(e1), wall)
    if world > 1:
        t = torch.tensor([ms], device=env.device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms / (calls * T)


def run_ours(args):
    import torch
    import torch.distributed as dist

    from collectivecrossing_b200 import BatchedCollectiveCrossing
    from collectivecrossing_b200.distributed import ShardedCollectiveCrossing

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly ONE JSON line: whatever libraries print while the job runs (NCCL's version
    # banner, ...) is sent to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    all_cpus = bind_to_gpu_numa_node(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    cfg = workload_config()
    n = args.envs
    A = 8
    # contiguous shard per rank; the RNG is keyed on the global env index (collectivecrossing_b200/distributed.py)
    sharded = ShardedCollectiveCrossing(cfg, n * world, seed=2026, device=dev, obs_dtype=args.obs_dtype, auto_reset=True)
    env = sharded.env
    assert sharded.count == n and sharded.offset == rank * n
    env.reset()
    desynchronise(env, torch)
    # steps per fused launch: at most --steps-per-launch, chosen so that the K timed steps are (almost) whole launches
    T = max(1, args.steps_per_launch)
    if T > 1:
        n_launch = max(1, -(-args.steps // T))
        T = max(1, args.steps // n_launch)
    # (the sampling thread starts before the warm-up: NVML's first queries can take longer than a whole timed region)
    sampler = ClockSampler(local) if rank == 0 else None
    for _ in range(args.warmup):
        env.step(policy=args.policy)
    traj = None
    if T > 1:   # allocates the [T, N, ...] output buffers, which every timed launch of T steps refills; warms the fused launch
        traj = env.rollout_trajectory(T, policy=args.policy)
    if world > 1:
        sharded.global_stats_device()                   # warms the NCCL communicator
    torch.cuda.synchronize()
    env.reset_stats()

    # the timed region (K steps) is repeated; the median repetition is the value, every repetition is reported
    reps = max(1, args.reps)
    rep_ms, stats_t, launches = [], None, 0
    if sampler:
        sampler.mark_begin()
    for _ in range(reps):
        launches0 = env.launch_count
        ms_r, stats_t = time_steps(env, torch, dist, args, args.steps, args.policy, world, T, sharded if world > 1 else None)
        launches = env.launch_count - launches0
        rep_ms.append(ms_r)
    if sampler:
        sampler.mark_end()
    clocks = sampler.stop() if sampler else None
    ms = median(rep_ms)
    env.check_error()
    kernel_name = env.last_kernel_name
    if args.dump_outputs and rank == 0:
        last = {"obs": env.obs, "reward": env.reward, "agent_flags": env.agent_flags, "env_flags": env.env_flags, "actions": env.actions_out}
        if T > 1 and args.steps % T == 0:   # the last timed step was the last step of a fused launch
            last = {k: None if traj[k] is None else traj[k][-1] for k in last}
        dump_outputs(args.dump_outputs, last, torch)

    # episode statistics of the job: at world > 1 the tensor the in-loop all-reduce left on the device
    st = sharded.stats_from_tensor(stats_t) if stats_t is not None else sharded.global_stats()
    collectives = (args.steps // T + args.steps % T if T > 1 else args.steps) if world > 1 else 0

    agent_steps = float(n) * A * args.steps * world
    value = agent_steps / (ms * 1e-3)
    peaks_path = ROOT / "MEASURED_PEAKS.json"
    if peaks_path.exists():
        peak, peak_src = float(json.loads(peaks_path.read_text())["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    else:
        peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
    # algorithmic bytes (SURVEY.md 8d): 12A+17+s_obs*A*(6+4A) per env-step of a single-step launch; a fused launch of T
    # steps keeps the state in registers, so its state term 2(3A+4)+8 is paid once per T steps
    b1 = env.algorithmic_bytes_per_env_step()
    bT = b1 - (2 * (3 * A + 4) + 8) * (1.0 - 1.0 / T)
    fused_steps = (args.steps // T) * T if T > 1 else 0
    total_bytes = (bT * fused_steps + b1 * (args.steps - fused_steps)) * n
    achieved = total_bytes / (ms * 1e-3) / 1e9
    traffic = None
    tp = ROOT / "profiles" / "traffic.json"
    if tp.exists():
        try:
            table = json.loads(tp.read_text())
            traffic = table.get(f"{args.obs_dtype}_{args.policy}_{n}_T{T}")
            if traffic is None and T > 1 and f"{args.obs_dtype}_{args.policy}_{n}_T20" in table:
                traffic = int(table[f"{args.obs_dtype}_{args.policy}_{n}_T20"] * T / 20)   # same kernel, same traffic per step
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "peak_source": peak_src, "kernel": kernel_name,
                "algorithmic_bytes_per_env_step": total_bytes / (n * args.steps), "steps_per_launch": T,
                "algorithmic_bytes_per_launch": bT * T * n if T > 1 else b1 * n,
                "formula": "12A+17+s_obs*A*(6+4A), A=8 (SURVEY.md 8d); in a fused launch of T steps the state term 2(3A+4)+8 is paid once per T steps"}

    # ---- e2e (headline): the reference's float32 rows in HOST buffers through the C ABI ----------------------------------
    # (the handle's own choice of row delivery: on a host with >= 8 threads the [A,4] table crosses PCIe and the float32 rows are
    #  rebuilt in the caller's buffer by the library's host threads; d2h_bytes_per_step is what the library copied)
    launches_before_e2e = env.launch_count
    host = env.make_host_buffers(pinned=True, actions_out=False)   # the caller supplies the actions: they are not copied back
    e2e_ms = time_e2e(env, torch, dist, world, args.policy, args.e2e_steps, host)
    call = env.last_host_call()
    rows_bytes = host["obs"].numel() * host["obs"].element_size()
    e2e = {"value": float(n) * A * world / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": call["h2d_bytes"],
           "d2h_bytes_per_step": call["d2h_bytes"] + n * A, "steps": args.e2e_steps, "ms_per_step": e2e_ms,
           "host_rows_bytes_per_step": rows_bytes, "expand_threads": call["expand_threads"], "chunks": call["chunks"],
           "path": "cc_policy_actions -> D2H actions (pinned) -> cc_step_host(H2D actions | fused step kernel | D2H "
                   + ("observation TABLE/reward/flags | float32 rows rebuilt in the caller's buffer by %d host threads (cc_set_host_expand: %s)"
                      % (call["expand_threads"], "this rank's share of the node's threads" if world > 1 else "the handle's automatic choice")
                      if call["expand_threads"] else "obs rows/reward/flags")
                   + ", chunks of envs pipelined over three streams); the caller receives the reference's float32 rows"}
    launches_e2e = env.launch_count - launches_before_e2e
    del host

    # ---- the same path with the other delivery formats of the SAME step (labelled, never the headline) ----------------------
    e2e_modes = {}
    if not args.no_extras:
        def mode(tag, obs, expand=None, T_=1, on_device=False, note=""):
            e = BatchedCollectiveCrossing(cfg, n, dev, seed=2026, global_env_offset=rank * n, obs_dtype=obs or "none", auto_reset=True)
            e.set_host_expand(expand if expand is not None else (sharded.host_threads or -2))
            e.reset()
            desynchronise(e, torch)
            # (a caller that supplies the actions does not need them copied back)
            h = e.make_host_buffers(pinned=True, n_steps=None if T_ == 1 else T_, actions_out=(T_ > 1 or on_device))
            ms_ = time_e2e(e, torch, dist, world, args.policy, max(args.e2e_steps, 2 * T_), h, T=T_, on_device_policy=on_device)
            c_ = e.last_host_call()
            e2e_modes[tag] = {"agent_steps_per_sec": float(n) * A * world / (ms_ * 1e-3), "ms_per_step": ms_,
                              "d2h_bytes_per_step": c_["d2h_bytes"] // T_ + (n * A if (T_ == 1 and not on_device) else 0),
                              "expand_threads": c_["expand_threads"], "vs_headline_e2e": e2e_ms / ms_, "note": note}
            e.close()
            del e, h
            torch.cuda.empty_cache()

        mode("float32_rows_over_pcie", "float32", expand=0, note="cc_set_host_expand(0): the float32 rows cross PCIe as the kernel wrote them (round 1's path, pipelined)")
        mode("table", "table", note="obs = compact table int8 [N,A,4] (CC_OBS_TABLE); rows on demand through cc_expand_obs_host")
        if world == 1:
            mode("int8_rows", "int8", note="obs = the reference's rows as int8 (rebuilt on the host from the table like the float32 rows; over PCIe: 6.8-7.2 ms)")
            mode("table_policy_on_device", "table", on_device=True, note="cc_step_host with the greedy policy in the kernel: no action round trip")
            mode("rollout_host_T8_table", "table", T_=8, note="cc_rollout_host: 8 steps per call, chunks stream out while the next chunk runs")
            mode("rollout_host_T8_float32", "float32", T_=8, note="cc_rollout_host: 8 steps per call, float32 rows")

    extras = {}
    if not args.no_extras:
        if world == 1:
            extras = secondary(args, torch, dist, cfg)
            try:   # BASELINE config 5's 1-GPU point: all 16.8 M envs on this GPU
                torch.cuda.empty_cache()
                extras.update(config5_sharded(args, torch, dist, cfg, world, rank, dev))
            except RuntimeError as exc:  # noqa: BLE001 - e.g. not enough free HBM next to another tenant: reported, not fatal
                extras["cfg5_16M_envs_waiting_sharded"] = {"error": str(exc)[:200]}
        else:
            extras = config5_sharded(args, torch, dist, cfg, world, rank, dev)

    if all_cpus:
        os.sched_setaffinity(0, all_cpus)
    if rank == 0:
        cpu = None
        if world == 1:
            cpu = cpu_python_loop(args, args.cpu_seconds)
            c_orc = cpu_c_oracle(args, min(4.0, args.cpu_seconds))
            cpu["c_oracle_openmp"] = {"value": c_orc["value"], "cores": c_orc["cores"], "sample": c_orc["sample"]}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8 (lattice cells, flag bytes; int32 step counters); rewards: f64 products rounded once to f32", "data": "synthetic",
            "config": config_dict(args, n * world), "clocks": clocks, "e2e": e2e, "gpu_launches": launches,
            "gpu_launches_e2e": launches_e2e, "roofline": roofline, "cpu_baseline": cpu,
            "repetitions": {"count": reps, "ms_per_region": rep_ms, "value": "median", "spread": (max(rep_ms) - min(rep_ms)) / ms},
            "collectives_in_timed_region": {"count": collectives, "what": "NCCL all-reduce (SUM) of the 8 episode statistics, one per launch, enqueued behind the kernel"},
            "episode_stats": st, "e2e_modes": e2e_modes, "host_copy_GBps": host_copy_bandwidth(torch) if world == 1 else None, "extras": extras,
        }
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def config5_sharded(args, torch, dist, cfg, world, rank, dev):
    """BASELINE config 5 as stated: 16,777,216 README envs sharded over the job's GPUs, waiting policy in the kernel, auto-reset,
    float32 rows, fused launches of 8 env-steps (2 on a single GPU) with ONE NCCL all-reduce of the episode statistics per launch
    inside the timed region at N > 1 (median of 3 regions of 5 launches; 10 on a single GPU)."""
    from collectivecrossing_b200.distributed import ShardedCollectiveCrossing

    # (on ONE GPU the [T, 16.8 M, 8, 38] float32 rows of a fused launch of 8 would be 163 GB: 2 steps per launch there)
    total, T, launches = 1 << 24, (8 if world > 1 else 2), (5 if world > 1 else 10)
    sh = ShardedCollectiveCrossing(cfg, total, seed=5, device=dev, obs_dtype="float32", auto_reset=True)
    env = sh.env
    env.reset()
    desynchronise(env, torch)
    for _ in range(30):
        env.step(policy="waiting")
    env.rollout_trajectory(T, policy="waiting")
    sh.global_stats_device()
    env.reset_stats()
    regions, stats_t = [], None
    for _ in range(3):
        ms, stats_t = time_steps(env, torch, dist, args, T * launches, "waiting", world, T, sh)
        regions.append(ms)
    ms = median(regions)
    st = sh.stats_from_tensor(stats_t)
    env.check_error()
    out = {"cfg5_16M_envs_waiting_sharded": {
        "agent_steps_per_sec": float(total) * 8 * T * launches / (ms * 1e-3), "ms_per_step": ms / (T * launches), "envs_total": total, "envs_per_gpu": sh.count,
        "n_gpus": world, "steps_per_launch": T, "ms_per_region": regions, "collectives_per_region": launches, "kernel": env.last_kernel_name,
        "episodes": st["episodes"], "episode_len_mean": st["episode_len_mean"], "terminated_fraction": st["terminated_fraction"],
        "algorithmic_GBps_per_gpu": (1329 - 64 * (1 - 1 / T)) * sh.count * T * launches / (ms * 1e-3) / 1e9}}
    env.close()
    return out


def secondary(args, torch, dist, cfg):
    """Secondary single-GPU measurements (reported under "extras", never as `value`): the other output modes / policies of the
    headline config (single-step launches, median of 3 regions), the lane-group mapping, small batches, and the shapes of BASELINE
    configs 3, 4 and 5 on one GPU.  `frac` = algorithmic bytes / time / the measured HBM peak."""
    from cases import large_config, readme_config

    from collectivecrossing_b200 import BatchedCollectiveCrossing

    out = {}
    dev = torch.device("cuda", torch.cuda.current_device())
    peaks_path = ROOT / "MEASURED_PEAKS.json"
    peak = float(json.loads(peaks_path.read_text())["hbm_gbs"]) if peaks_path.exists() else 6650.0
    M = 1 << 20
    binary = readme_config("binary", "individual", 100, goal_reward=1.0, no_goal_reward=0.0)
    constneg = readme_config("constant_negative", "individual", 100, step_penalty=-1.0)
    runs = (
        # tag, config, envs, obs dtype, policy, kernel, timed steps per region, steps per launch
        ("1M_envs_fp32_greedy_single_step_launches", cfg, M, "float32", "greedy", "auto", 50, 1),
        ("1M_envs_int8_greedy", cfg, M, "int8", "greedy", "auto", 50, 1),
        ("1M_envs_int8_greedy_fused20", cfg, M, "int8", "greedy", "auto", 40, 20),
        ("1M_envs_table_greedy", cfg, M, "table", "greedy", "auto", 50, 1),
        ("1M_envs_noobs_greedy", cfg, M, "none", "greedy", "auto", 50, 1),
        ("1M_envs_noobs_greedy_fused20", cfg, M, "none", "greedy", "auto", 40, 20),
        ("1M_envs_int8_waiting", cfg, M, "int8", "waiting", "auto", 50, 1),
        ("1M_envs_fp32_waiting", cfg, M, "float32", "waiting", "auto", 50, 1),
        ("1M_envs_fp32_random", cfg, M, "float32", "random", "auto", 50, 1),
        ("1M_envs_fp32_greedy_lane_group_kernel", cfg, M, "float32", "greedy", "lanes", 50, 1),
        ("cfg2_65536_envs_fp32_greedy", cfg, 65536, "float32", "greedy", "auto", 100, 1),
        ("cfg2_65536_envs_fp32_greedy_fused20", cfg, 65536, "float32", "greedy", "auto", 200, 20),
        ("cfg4_binary_individual_4M_envs_fp32_random", binary, 4 * M, "float32", "random", "auto", 10, 1),
        ("cfg4_constant_negative_individual_4M_envs_fp32_random", constneg, 4 * M, "float32", "random", "auto", 10, 1),
        ("cfg5_shard_2M_envs_fp32_waiting", cfg, 2 * M, "float32", "waiting", "auto", 20, 1),
        ("cfg3_64x32_64agents_simple_distance_all_1M_envs_int8_random", large_config(512), M, "int8", "random", "auto", 5, 1),
        ("cfg3_64x32_64agents_simple_distance_all_1M_envs_fp32_random", large_config(512), M, "float32", "random", "auto", 3, 1),
    )
    # fused multi-step launches of the headline kernel at other lengths (first: before the 20-70 GB allocations of configs 3-5) (the state term 2(3A+4)+8 is paid once per T steps)
    for T, n_envs in ((4, M), (16, M)):
        env = BatchedCollectiveCrossing(cfg, n_envs, dev, seed=1, obs_dtype="float32", auto_reset=True)
        env.reset()
        desynchronise(env, torch)
        env.rollout_trajectory(T, policy="greedy")
        regions = [time_steps(env, torch, dist, args, 12 * T, "greedy", 1, T)[0] / (12 * T) for _ in range(3)]
        ms = median(regions)
        env.check_error()
        a = env.num_agents
        bytes_step = a + (2 * (3 * a + 4) + 8) / T + 5 * a + 1 + 4 * a * (6 + 4 * a)
        out[f"fused_rollout_T{T}_1M_envs_fp32_greedy"] = {
            "agent_steps_per_sec": n_envs * a / (ms * 1e-3), "ms_per_step": ms, "algorithmic_GBps": bytes_step * n_envs / (ms * 1e-3) / 1e9,
            "frac": bytes_step * n_envs / (ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_env_step": bytes_step, "kernel": env.last_kernel_name,
            "agents_per_env": a, "envs": n_envs, "steps_per_launch": T}
        env.close()
        del env
        torch.cuda.empty_cache()
    for tag, c, n, obs, pol, kern, steps, T in runs:
        env = BatchedCollectiveCrossing(c, n, dev, seed=1, obs_dtype=obs, auto_reset=True, kernel=kern)
        env.reset()
        desynchronise(env, torch)
        for _ in range(5):
            env.step(policy=pol)
        if T > 1:
            env.rollout_trajectory(T, policy=pol)
        regions = [time_steps(env, torch, dist, args, steps, pol, 1, T)[0] for _ in range(3)]
        ms = median(regions)
        env.check_error()
        a = env.num_agents
        b1 = env.algorithmic_bytes_per_env_step()
        bT = b1 - (2 * (3 * a + 4) + 8) * (1.0 - 1.0 / T)
        gbs = bT * n / (ms / steps * 1e-3) / 1e9
        out[tag] = {"agent_steps_per_sec": n * a * steps / (ms * 1e-3), "ms_per_step": ms / steps, "algorithmic_GBps": gbs, "frac": gbs / peak,
                    "algorithmic_bytes_per_env_step": bT, "kernel": env.last_kernel_name, "agents_per_env": a, "envs": n, "steps_per_launch": T,
                    "ms_per_region": regions}
        env.close()
        del env
        torch.cuda.empty_cache()

    return out


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
