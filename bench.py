#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 IndustrialEnv step path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[1]): ChemicalReactor-v0, 65,536 envs PER GPU, fp32. One bench "step" is one
1,000-env-step pass over every env of the rank's shard through the fused K=64 rollout kernel (15 x 64 + 40 =
16 launches), with the reference harness's policy (uniform-random actions = action_space.sample(),
performance_benchmark.py:106-133) and process noise drawn in-kernel (Philox) and auto-reset on done.
value = env-steps/s summed over ranks (weak scaling: the per-GPU shard is fixed; shards are keyed by global env
id, no inter-GPU traffic while stepping, one NCCL all-reduce of the counters at the end of the timed region).

Also measured in the same run and reported in the JSON line:
  roofline      -- the kernel dominating the timed region (fused rollout): algorithmic fp32 ops / s vs the fp32
                   non-FMA issue peak measured live with a probe kernel (the path is element-wise ODE integration).
  single_step   -- the single-step kernel: env-steps/s at 65,536 envs (launch-bound) and its HBM roofline at 4M envs
                   (state larger than L2), achieved GB/s vs MEASURED_PEAKS.json.
  e2e           -- env.rollout(1000, "random", init_states=host) -> host returns / violations / obs: the same workload
                   through the drop-in API with host buffers (nig_rollout_host); e2e_step_api = one env.step() per call.
  cpu_baseline  -- the reference's own Python step loop (performance_benchmark.py:106-133, unmodified modules from
                   oracle/_ref) on one core and on all host cores, plus the C oracle port, in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "neorl-industrial-gym_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

ENVS_PER_GPU = 65536
HORIZON = 1000            # env-steps per env per bench step
K = 64                    # fused steps per launch
METRIC = "env-steps/sec (ChemicalReactor-v0, 64K envs)"
UNIT = "env-steps/s"
ALG_BYTES_PER_STEP = 122  # SURVEY section 8d: 48 state r + 48 state w + 12 action + 4 reward + 2 flags + 8 counter r/w
ALG_OPS_PER_STEP = 128    # SURVEY section 8d: dynamics 76 + reward 30 + step logic 22 (RNG / addressing excluded)
WORKLOAD = ("ChemicalReactor-v0 batched 65,536 envs x 1,000 steps fp32 per GPU; fused K=64 rollout kernel "
            "(15x64+40), in-kernel uniform-random policy (= action_space.sample()), Philox process noise, auto-reset")


def launches_per_pass():
    return (HORIZON + K - 1) // K


class ClockSampler:
    """SM clock / throttle reasons sampled IN PROCESS through NVML (nvidia-ml-py) every ~1 ms from before the warm-up until
    after the timed region; stop(t0, t1) keeps the samples taken inside [t0, t1] (perf_counter times) -- a 13 ms timed region
    still gets a dozen samples, which a 50 ms nvidia-smi poll never saw."""
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index: int):
        self.index, self.rows, self.stop_flag, self.thread, self.err = index, [], False, None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
        except Exception as ex:          # no NVML: the driver's own clock record is the one that counts
            self.err = repr(ex)

    def _poll(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                why = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((time.perf_counter(), float(mhz), int(why)))
            except Exception as ex:
                self.err = repr(ex)
                return
            time.sleep(0.001)

    def stop(self, t0: float, t1: float):
        self.stop_flag = True
        if self.thread is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [f"NVML unavailable: {self.err}"], "samples": 0}
        self.thread.join(timeout=1.0)
        inside = [r for r in self.rows if t0 <= r[0] <= t1]
        scope = "timed region"
        if not inside:                   # (cannot happen with a >= 3 ms region; kept so the key is never silently empty)
            inside, scope = self.rows[-20:], "last samples before the end of the timed region"
        reasons = sorted({name for _, _, why in inside for name, bit in self.REASONS if why & bit})
        return {"sm_mhz": float(np.median([r[1] for r in inside])) if inside else None, "sm_max_mhz": self.max_mhz,
                "reasons": reasons, "samples": len(inside), "scope": scope, "source": "NVML in-process, 1 ms period"}


def issued_per_warp_step():
    """Executed warp-instructions per warp per step of the fused reactor kernel, read from the committed ncu source summary of
    the current build (profiles/r02_*_reactor_rollout_kernel_source_summary.txt, newest first) -- not a constant in this file."""
    import glob
    import re
    for path in sorted(glob.glob(os.path.join(ROOT, "profiles", "r0*_reactor_rollout_kernel_source_summary.txt")), reverse=True):
        try:
            m = re.search(r"total executed warp-instructions \d+\s+\(([0-9.]+) per unit\)", open(path).read())
            if m:
                return float(m.group(1)), os.path.relpath(path, ROOT)
        except OSError:
            pass
    return None, None


def ncu_traffic(key_prefix: str):
    """DRAM bytes per launch of a kernel from the committed ncu --set full capture (profiles/r02_traffic.json, else r01), or None."""
    try:
        path = os.path.join(ROOT, "profiles", "r02_traffic.json")
        if not os.path.exists(path):
            path = os.path.join(ROOT, "profiles", "r01_traffic.json")
        with open(path) as f:
            d = json.load(f)
        for k, v in d.items():
            if k.startswith(key_prefix):
                return v["dram_bytes_per_launch"]
    except Exception:
        pass
    return None


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------ CPU arms
def host_threads() -> int:
    """Host cores this process may use (torchrun exports OMP_NUM_THREADS=1; the oracle takes an explicit thread count)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_rollout_rate(n_envs: int, horizon: int, threads: int, seed: int = 0):
    from oracle import oracle as O
    env = O.OracleEnv(O.REACTOR, n_envs, seed=seed, exp_mode=0, threads=threads)
    env.reset()
    t0 = time.perf_counter()
    O.rollout(env, horizon, O.POLICY_UNIFORM)
    dt = time.perf_counter() - t0
    return n_envs * horizon / dt, dt


def bench_config(world: int):
    """`config` of the JSON line -- the SAME object in the CUDA arm and the reference arm (what differs between the arms,
    e.g. the reference arm's bounded sample or the CUDA arm's launch counts, is reported outside it)."""
    return {"workload": WORKLOAD, "envs_per_gpu": ENVS_PER_GPU, "steps_per_env_per_bench_step": HORIZON, "K": K,
            "parallelism": f"env-index shards x{world}, no data-path collective",
            "l2": "256 MiB write between timed iterations (outside the CUDA-event brackets); state lives in registers across K steps"}


def reference_loop(mode: str, procs: int = 0, repeats: int = 5, rounds: int = 1, timeout: float = 600.0):
    """The reference's own step loop (performance_benchmark.py:106-133, unmodified modules from oracle/_ref) timed by
    oracle/ref_bench.py in a process of its own; None when oracle/_ref did not travel to this machine."""
    cmd = [sys.executable, os.path.join(ROOT, "oracle", "ref_bench.py"), "--mode", mode, "--steps", str(HORIZON),
           "--repeats", str(repeats), "--rounds", str(rounds)]
    if procs:
        cmd += ["--procs", str(procs)]
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout)
        return json.loads(r.stdout.strip().splitlines()[-1])
    except Exception:
        return None


def port_baseline(budget_s: float):
    """The C oracle port (scalar per env, same workload incl. RNG) on all host threads; bounded sample."""
    threads = host_threads()
    r1, _ = cpu_rollout_rate(2048, 250, 1)                       # calibrate (single thread)
    n = int(min(ENVS_PER_GPU, max(1024, r1 * threads * 0.5 * budget_s / HORIZON))) // 256 * 256 or 256
    rate, dt = cpu_rollout_rate(n, HORIZON, threads)
    return {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"C oracle port (oracle/nig_oracle.c, scalar per env, same policy / noise / auto-reset), {n} envs x {HORIZON} "
                      f"steps in {dt:.2f} s on {threads} threads; single-thread rate {r1:.3g} env-steps/s"}


def cpu_baseline(budget_s: float = 8.0):
    """The reference's own CPU step loop on this box's host cores, in the same run: (i) one core, median of 5 x 1,000 steps;
    (ii) P = all usable cores, P forked processes with one env each (the reference has no batched / jit / vmap path);
    plus, labelled as ours, the C oracle port on all threads."""
    threads = host_threads()
    port = port_baseline(budget_s)
    single = reference_loop("single", repeats=5)
    if single is None:
        port["note"] = "oracle/_ref (the reference's modules, oracle/make_ref.py) is not present on this machine: C port only"
        return port
    reps = max(1, int(round(single["steps_per_sec"] * 0.6 * budget_s / HORIZON)))
    allc = reference_loop("all", procs=threads, repeats=reps, rounds=1)
    return {"value": allc["steps_per_sec"], "unit": UNIT, "cores": threads, "kind": "reference",
            "sample": f"the reference's own loop (performance_benchmark.py:106-133; unmodified environments/*.py + core/types.py "
                      f"from oracle/_ref, gymnasium / jax stubbed, numpy {single['numpy']}): {threads} forked processes x 1 env x "
                      f"{reps} x {HORIZON} steps in {allc['round_wall_s'][0]:.2f} s. The reference has no batched / jit / vmap path.",
            "single_core": {"value": single["steps_per_sec"], "unit": UNIT, "cores": 1, "min": single["min"], "max": single["max"],
                            "sample": f"median of {single['repeats']} x {HORIZON} steps, one env, one core"},
            "port": port}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path -- its per-env Python step loop
    (performance_benchmark.py:106-133) from oracle/_ref -- on all host cores (one forked process per core, one env each);
    each bench step is a bounded sample of the 65,536 x 1,000 workload (~1 s). Falls back to the C port (kind "port")
    only if oracle/_ref is absent."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = host_threads()
    single = reference_loop("single", repeats=3)
    if single is not None:
        reps = max(1, int(round(single["steps_per_sec"] * 0.6 * 1.0 / HORIZON)))
        res = reference_loop("all", procs=threads, repeats=reps, rounds=args.warmup + args.steps)
        walls = res["round_wall_s"][args.warmup:]
        per_step = threads * reps * HORIZON
        dt = sum(walls)
        kind = "reference"
        sample = (f"the reference's own loop (performance_benchmark.py:106-133, unmodified modules from oracle/_ref): per bench step "
                  f"{threads} forked processes x 1 env x {reps} x {HORIZON} steps = {per_step} env-steps; single core "
                  f"{single['steps_per_sec']:.0f} steps/s")
    else:
        r1, _ = cpu_rollout_rate(2048, 250, 1)
        n = int(min(ENVS_PER_GPU, max(1024, r1 * threads * 0.5 * 1.0 / HORIZON))) // 256 * 256 or 256
        for _ in range(args.warmup):
            cpu_rollout_rate(n, HORIZON, threads)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            cpu_rollout_rate(n, HORIZON, threads)
        dt = time.perf_counter() - t0
        per_step = n * HORIZON
        kind = "port"
        sample = f"C oracle port, {n} envs x {HORIZON} steps per bench step, {threads} threads (oracle/_ref absent on this machine)"
    value = per_step * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(args.gpus),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample,
                         "env_steps_per_bench_step": per_step},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ GPU arm
def run_gpu(args):
    import torch
    import neorl_industrial as ni
    from neorl_industrial import _native as N

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    hbm_peak, peak_src = measured_peaks()

    n = ENVS_PER_GPU
    env = ni.NativeEnv(N.ENV_CHEMICAL_REACTOR, n, device=local, seed=args.seed, env_id_offset=rank * n)
    env.reset_device()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2

    def one_pass():
        # 1,000 steps as 15 x K=64 + one K=40 fused launches per env slice (C ABI nig_rollout_steps: the slices advance on
        # internal streams forked from / joined to the current stream, so the CUDA events below bracket all of them)
        env.rollout_steps_device(HORIZON, K, N.POLICY_UNIFORM)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    from neorl_industrial.distributed import allreduce_device_stats
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        one_pass()
    if dist is not None:
        allreduce_device_stats(env)               # (warm-up of the communicator / the grouped all-reduce)
    barrier()
    env.clear_stats()
    launches0 = env.launch_count
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    t_wall0 = time.perf_counter()
    for i in range(args.steps):
        flush.fill_(i & 0xFF)                     # L2 flush between timed iterations (outside the event brackets)
        ev[i][0].record()
        one_pass()
        ev[i][1].record()
    # the path's only collective, inside the timed region: counters / sums / extrema of all shards in ONE grouped NCCL launch
    # through the C ABI (nig_allreduce_stats) on this stream, bracketed by its own events and added to the step times
    ar0, ar1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ar0.record()
    if dist is not None:
        allreduce_device_stats(env)
    ar1.record()
    barrier()
    t_wall1 = time.perf_counter()
    t_wall = t_wall1 - t_wall0
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    launches = env.launch_count - launches0
    step_ms = [a.elapsed_time(b) for a, b in ev]
    allreduce_ms = ar0.elapsed_time(ar1) if dist is not None else 0.0
    total_ms = torch.tensor([sum(step_ms) + allreduce_ms], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms.item())
    ar_max = torch.tensor([allreduce_ms], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(ar_max, op=dist.ReduceOp.MAX)
    allreduce_us = float(ar_max.item()) * 1e3
    value = world * n * HORIZON * args.steps / (total_ms * 1e-3)
    counters, fsum = env.read_stats()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, env, counters, fsum)

    extra = {}
    e2e = None
    if "e2e" in args.sections:
        e2e = e2e_rollout(ni, n, local, rank, world, max(3, min(args.steps, 100)), args.warmup, args.seed, dist, torch)
    others = other_configs(torch, ni, N, local, rank, world, dist, args.seed) if "configs" in args.sections else None
    if rank == 0:
        if e2e is not None:
            extra["e2e"] = e2e
        if others is not None:
            extra["other_configs"] = others
        # ---- roofline of the dominant kernel of the timed region (fused rollout): fp32 pipe
        # per whole-population K-step launch (15 x K=64 and one K=40 per bench step). The env slices of nig_rollout_steps
        # run these launches concurrently on several streams, so the duration is the step time shared out over them
        kernel_ms = (total_ms - allreduce_us * 1e-3) / (args.steps * launches_per_pass())
        issued, issued_src = issued_per_warp_step()
        ops_per_launch = ALG_OPS_PER_STEP * n * HORIZON / launches_per_pass()
        import ctypes as C
        ops = C.c_double(0)
        st = int(torch.cuda.current_stream().cuda_stream)
        N.check(N.lib().nig_fp32_probe(local, 200, C.byref(ops), st))
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        N.check(N.lib().nig_fp32_probe(local, 20000, C.byref(ops), st))
        e1.record()
        torch.cuda.synchronize()
        fp32_peak = ops.value / (e0.elapsed_time(e1) * 1e-3) / 1e12     # T op/s, unfused add/mul, measured live
        achieved = ops_per_launch / (kernel_ms * 1e-3) / 1e12
        extra["roofline"] = {
            "kernel": "rollout_kernel<Reactor, default constraints, POLICY_UNIFORM> (K=64 fused steps)",
            "bound": "fp32", "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s", "frac": achieved / fp32_peak,
            "traffic": ncu_traffic("rollout_kernel<Reactor"),
            "ncu": issued_src,
            # every instruction the kernel issues (the ncu count of the committed source summary) against one warp-instruction
            # per cycle per SM sub-partition at the peak the probe measured: how full the issue slots are over the whole launch
            "issued_per_warp_step": issued,
            "issue_slot_frac": (issued / ALG_OPS_PER_STEP * achieved / fp32_peak) if issued else None,
            "note": f"algorithmic {ALG_OPS_PER_STEP} fp32 ops/env-step (SURVEY 8d; RNG, IEEE-division expansion and addressing "
                    "excluded) x env-steps per launch / mean launch time (issue_slot_frac counts every issued instruction, RNG included); "
                    "peak = unfused FADD/FMUL issue rate measured live by nig_fp32_probe (nominal 148 SM x 128 lanes x 1.965 GHz = "
                    "37.2 T op/s). Tensor cores do not apply: element-wise ODE.",
        }
        # ---- single-step kernel at 65,536 envs (launch-bound) and its HBM roofline at 4M envs (> L2)
        if "single" in args.sections:
            extra["single_step"] = single_step_section(torch, ni, N, local, dev, flush, hbm_peak, peak_src, args)
            # BASELINE.json's metric asks for "% HBM roofline": that is the single-step kernel's (the fused kernel above
            # is FP32-issue bound and moves 60 B per env per 64 steps); repeated at the top level next to `roofline`
            extra["roofline_hbm"] = extra["single_step"]["roofline"]
            extra["actions_tma"] = actions_section(torch, ni, N, local, dev, args)
        # ---- e2e through the Python drop-in API with host buffers
        if "e2e" in args.sections:
            extra["e2e_step_api"] = e2e_step_api(ni, n, local, args)
            extra["torch_step_api"] = torch_api(torch, ni, n, local, args)
        if "cpu" in args.sections:
            extra["cpu_baseline"] = cpu_baseline()
    if dist is not None:
        dist.barrier()
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": bench_config(world),
        "launch_config": {"launches_per_bench_step": int(launches) // max(args.steps, 1),
                          "env_slices_per_gpu": (int(launches) // max(args.steps, 1)) // launches_per_pass()},
        "clocks": clocks, "gpu_launches": int(launches), "allreduce_us": allreduce_us,
        "wall_s_timed_region": t_wall,
        "counters": {"steps": int(counters[0]), "episodes": int(counters[1]), "violations": int(counters[5]),
                     "critical_shutdowns": int(counters[4]), "return_sum": float(fsum[0])},
    }
    line.update(extra)
    print(json.dumps(line), flush=True)
    if dist is not None:
        dist.destroy_process_group()


def dump_outputs(out_dir, env, counters, sums):
    """--dump-outputs DIR: what the timed path hands its caller after the last timed step, as DIR/<name>.npy -- the env
    state of rank 0's shard (observation float32 [n, 12]; episode step, episode violation count and done flag as float64
    [n]) and the stats block over the timed steps (counters and sums, float64; all-reduced when there are several ranks). About 5 MB at
    65,536 envs. The inputs depend only on the arguments (seed, warm-up and step counts), so two builds run with the same
    arguments can be compared array by array: bit for bit, except the fp64 sums, which the kernels accumulate with
    atomics in no fixed order (their last bits vary from run to run)."""
    os.makedirs(out_dir, exist_ok=True)
    state, ep_step, ep_viol, done = env.get_state_host()
    arrays = {"obs": state, "episode_step": ep_step.astype(np.float64), "episode_violations": ep_viol.astype(np.float64),
              "done": done.astype(np.float64), "stats_counters": counters.astype(np.float64), "stats_sums": sums}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def single_step_section(torch, ni, N, local, dev, flush, hbm_peak, peak_src, args):
    out = {}
    # (a) the BASELINE config: 65,536 envs x 1,000 single-step launches, device-resident SoA actions
    env = ni.NativeEnv(N.ENV_CHEMICAL_REACTOR, ENVS_PER_GPU, device=local, seed=args.seed)
    env.reset_device()
    acts = torch.rand((3, env.pitch), device=dev) * 2 - 1
    rew, fl, vm = env.empty(), env.empty(dtype=torch.uint8), env.empty(dtype=torch.uint8)
    for _ in range(50):
        env.step_device(acts, reward=rew, flags=fl, viol_mask=vm)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(HORIZON):
        env.step_device(acts, reward=rew, flags=fl, viol_mask=vm)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    frac64 = lambda us: ALG_BYTES_PER_STEP * ENVS_PER_GPU / (us * 1e-6) / 1e9 / hbm_peak
    out["envs_64k"] = {"value": ENVS_PER_GPU * HORIZON / (ms * 1e-3), "unit": UNIT, "us_per_launch": ms * 1e3 / HORIZON,
                       "hbm_frac": frac64(ms * 1e3 / HORIZON),
                       "note": "1,000 back-to-back launches; 8 MB working set is L2-resident, launch-latency bound"}
    # the same 1,000 launches as 10 replays of a captured 100-launch CUDA graph (device-resident tick: fresh noise each step)
    try:
        env.use_device_tick(2)                   # device base + per-launch sequence offsets (nig_use_device_tick mode 2)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            for _ in range(100):
                env.step_device(acts, reward=rew, flags=fl, viol_mask=vm)
            env.commit_ticks()                   # last node: the base moves on by 100 per replay
        g.replay()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(HORIZON // 100):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        msg = e0.elapsed_time(e1)
        out["envs_64k_cuda_graph"] = {"value": ENVS_PER_GPU * HORIZON / (msg * 1e-3), "unit": UNIT, "us_per_launch": msg * 1e3 / HORIZON,
                                      "hbm_frac": frac64(msg * 1e3 / HORIZON),
                                      "note": "10 replays of a 100-launch CUDA graph (nig_use_device_tick mode 2 + nig_commit_ticks; programmatic dependent launch)"}
        # the same replay without the device counter block (nig_track_step_stats(env, 0): IndustrialEnv.step has no global counters;
        # its per-env outputs are complete) and without the return accumulator: what the plain gym loop needs
        env.track_step_stats(False)
        env.track_returns(False)
        g2 = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g2):
            for _ in range(100):
                env.step_device(acts, reward=rew, flags=fl, viol_mask=vm)
            env.commit_ticks()
        g2.replay()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(HORIZON // 100):
            g2.replay()
        e1.record()
        torch.cuda.synchronize()
        msq = e0.elapsed_time(e1)
        out["envs_64k_cuda_graph_no_counters"] = {"value": ENVS_PER_GPU * HORIZON / (msq * 1e-3), "unit": UNIT, "us_per_launch": msq * 1e3 / HORIZON,
                                                  "hbm_frac": frac64(msq * 1e3 / HORIZON),
                                                  "note": "as above with nig_track_step_stats(env, 0) and nig_track_returns(env, 0): no warp reductions / "
                                                          "atomics at the tail of the launch, no 16 B of accumulator traffic"}
    except Exception as ex:                                   # graph capture is an optimisation, never a requirement
        out["envs_64k_cuda_graph"] = {"error": repr(ex)}
    env.close()
    # (b) HBM roofline: 16,777,216 envs (2 GB of state + io per launch, >> L2; the copy that MEASURED_PEAKS.json times
    # moves 4 GB), in-kernel Philox noise, auto-reset
    n_big = 1 << 24
    env = ni.NativeEnv(N.ENV_CHEMICAL_REACTOR, n_big, device=local, seed=args.seed)
    env.track_returns(False)       # the plain gym step loop (performance_benchmark.py:106-133): no per-env return accumulator;
    env.reset_device()             # the default (tracking on, 16 B more per env-step) is measured next to it below
    acts = torch.rand((3, env.pitch), device=dev) * 2 - 1
    rew, fl, vm = env.empty(), env.empty(dtype=torch.uint8), env.empty(dtype=torch.uint8)
    for _ in range(10):                                    # 640 steps: past the first wave of episode ends, so that the
        env.rollout_device(64, N.POLICY_UNIFORM)           # timed launches see the steady-state mix (auto-resets firing)
    for _ in range(5):
        env.step_device(acts, reward=rew, flags=fl, viol_mask=vm)
    torch.cuda.synchronize()
    reps = 30
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in evs:
        a.record()
        env.step_device(acts, reward=rew, flags=fl, viol_mask=vm)
        b.record()
    torch.cuda.synchronize()
    ms = float(np.mean([a.elapsed_time(b) for a, b in evs]))
    gbs = ALG_BYTES_PER_STEP * n_big / (ms * 1e-3) / 1e9
    out["roofline"] = {"kernel": "step_pipe_kernel<Reactor, VEC=2, default constraints> (persistent, cp.async.bulk 3-stage ring)", "bound": "hbm", "achieved": gbs,
                       "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak, "traffic": ncu_traffic("step_pipe_kernel<Reactor"), "peak_source": peak_src,
                       "envs": n_big, "ms_per_launch": ms, "value": n_big / (ms * 1e-3),
                       "note": f"{ALG_BYTES_PER_STEP} algorithmic B/env-step x {n_big} envs per launch / mean launch time; inputs larger than L2; "
                               "steady-state episode mix (640 fused warm-up steps first: 0.25 % of the envs auto-reset per step); "
                               "nig_track_returns(env, 0): the per-env episode-return accumulator is not part of the 122 B"}
    env.track_returns(True)
    for a, b in evs:
        a.record()
        env.step_device(acts, reward=rew, flags=fl, viol_mask=vm)
        b.record()
    torch.cuda.synchronize()
    ms_t = float(np.mean([a.elapsed_time(b) for a, b in evs]))
    out["roofline_with_return_tracking"] = {"ms_per_launch": ms_t, "value": n_big / (ms_t * 1e-3),
                                            "achieved_138B": (ALG_BYTES_PER_STEP + 16) * n_big / (ms_t * 1e-3) / 1e9,
                                            "frac_138B": (ALG_BYTES_PER_STEP + 16) * n_big / (ms_t * 1e-3) / 1e9 / hbm_peak,
                                            "note": "default handle: + 8 B read + 8 B write of the fp64 episode-return accumulator per env-step"}
    env.close()
    return out


def actions_section(torch, ni, N, local, dev, args):
    """north_star (2): action SEQUENCES staged in shared memory via TMA. 65,536 envs x 1,000 steps with teacher-forced actions
    from a device tensor [K = 64][A = 3][pitch] (12 B of HBM per env-step instead of the in-kernel policy's draw), process noise
    in-kernel: the cp.async.bulk.tensor.3d flavour (16-step boxes, double-buffered, mbarrier) against the flavour that
    prefetches the next step's actions into registers with LDG."""
    n = ENVS_PER_GPU
    env = ni.NativeEnv(N.ENV_CHEMICAL_REACTOR, n, device=local, seed=args.seed)
    acts = torch.rand((K, 3, env.pitch), device=dev) * 2 - 1
    out = {"workload": f"ChemicalReactor-v0, {n} envs x {HORIZON} steps, K = {K} per launch, actions [K][3][pitch] fp32 on the device"}
    for name, tma in (("tma_3d", True), ("ldg_register_prefetch", False)):
        env.reset_device()

        def one_pass():
            done = 0
            while done < HORIZON:
                k = min(K, HORIZON - done)
                env.rollout_device(k, N.POLICY_ACTIONS, actions=acts, use_tma=tma)
                done += k
        for _ in range(3):
            one_pass()
        torch.cuda.synchronize()
        ts = []
        for _ in range(7):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); one_pass(); e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        ms = float(np.median(ts))
        out[name] = {"value": n * HORIZON / (ms * 1e-3), "unit": UNIT, "ms_per_1000_steps": ms,
                     "kernel": "rollout_kernel<Reactor, default constraints, POLICY_ACTIONS, TMA=%s>" % ("true" if tma else "false")}
    env.close()
    return out


def other_configs(torch, ni, N, local, rank, world, dist, seed):
    """The remaining BASELINE.json configs, measured briefly (device-resident, CUDA events, max over ranks):
    configs[2] PowerGrid-v0 1,048,576 envs sharded over the ranks, fused K=64 rollout + single-step kernel, auto-reset;
    configs[3] ChemicalReactor-v0 + SafetyWrapper temperature / pressure bands, counters NCCL all-reduced;
    configs[4] (rank 0) 1M-transition 'mixed' dataset written on the device in D4RL layout + pinned export."""
    from neorl_industrial.distributed import allreduce_device_stats, shard_bounds
    from neorl_industrial.safety import BoundConstraint, SafetyWrapper
    dev = torch.device("cuda", local)
    out = {}

    def timed(fn, reps):
        for _ in range(3):                 # warm-up (nig_rollout_steps captures its launch sequence on the second identical call)
            fn()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / reps

    def graph_step_ms(env, acts, rew, fl, vm, launches=50, replays=4):
        """One IndustrialEnv.step per launch as replays of a captured `launches`-launch CUDA graph (sequence ticks + programmatic
        dependent launch): the host thread (a Python call per launch, W processes per box) no longer paces a shard's step."""
        try:
            env.use_device_tick(2)
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                env.step_device(acts, reward=rew, flags=fl, viol_mask=vm)
            torch.cuda.current_stream().wait_stream(side)
            env.commit_ticks()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                for _ in range(launches):
                    env.step_device(acts, reward=rew, flags=fl, viol_mask=vm)
                env.commit_ticks()
            ms = timed(g.replay, replays) / launches
            env.use_device_tick(False)
            return ms
        except Exception as ex:                                   # graph capture is an optimisation, never a requirement
            sys.stderr.write(f"graph_step_ms: {ex!r}\n")
            try:
                env.use_device_tick(False)
            except Exception:
                pass
            return None

    # ---- configs[2]: PowerGrid-v0, 1M envs over the ranks
    n_total = 1 << 20
    off, cnt = shard_bounds(n_total, world, rank)
    env = ni.NativeEnv(N.ENV_POWER_GRID, cnt, device=local, seed=seed, env_id_offset=off)
    env.reset_device()
    ms = timed(lambda: env.rollout_steps_device(256, 64, N.POLICY_UNIFORM), 3)
    acts = torch.rand((8, env.pitch), device=dev) * 2 - 1
    rew, fl, vm = env.empty(), env.empty(dtype=torch.uint8), env.empty(dtype=torch.uint8)
    ms1e = timed(lambda: env.step_device(acts, reward=rew, flags=fl, viol_mask=vm), 20)
    ms1g = graph_step_ms(env, acts, rew, fl, vm)
    ms1 = min(ms1e, ms1g) if ms1g else ms1e
    view = allreduce_device_stats(env)
    torch.cuda.synchronize()
    st = env.stats_dict()
    hbm_peak, _ = measured_peaks()
    out["powergrid_1m"] = {
        "workload": f"PowerGrid-v0 (32-d state, 8-d action, 23 Gaussian draws/step), {n_total} envs over {world} rank(s), auto-reset",
        "rollout_k64": {"value": n_total * 256 / (ms * 1e-3), "unit": UNIT, "ms_per_256_steps": ms},
        "single_step": {"value": n_total / (ms1 * 1e-3), "unit": UNIT, "ms_per_launch": ms1,
                        "ms_per_launch_eager": ms1e, "ms_per_launch_graph_replay": ms1g,
                        "hbm_frac_per_gpu": 302 * cnt / (ms1 * 1e-3) / 1e9 / hbm_peak,
                        "note": "302 algorithmic B/env-step; the 23 in-kernel Gaussian draws per step make this kernel issue-bound, not HBM-bound"},
        "allreduced": {"steps": st["steps"], "episodes": st["episodes"], "violations": st["violations"]}}
    env.close()
    # ---- RobotAssembly-v0 (the third env implemented upstream), same sharding
    env = ni.NativeEnv(N.ENV_ROBOT_ASSEMBLY, cnt, device=local, seed=seed, env_id_offset=off)
    env.reset_device()
    ms = timed(lambda: env.rollout_steps_device(256, 64, N.POLICY_UNIFORM), 3)
    acts = torch.rand((7, env.pitch), device=dev) * 2 - 1
    ms1e = timed(lambda: env.step_device(acts, reward=rew, flags=fl, viol_mask=vm), 20)
    ms1g = graph_step_ms(env, acts, rew, fl, vm)
    ms1 = min(ms1e, ms1g) if ms1g else ms1e
    out["robot_assembly_1m"] = {
        "workload": f"RobotAssembly-v0 (24-d state, 7-d action, fp64 kinematics), {n_total} envs over {world} rank(s), auto-reset",
        "rollout_k64": {"value": n_total * 256 / (ms * 1e-3), "unit": UNIT, "ms_per_256_steps": ms},
        "single_step": {"value": n_total / (ms1 * 1e-3), "unit": UNIT, "ms_per_launch": ms1,
                        "ms_per_launch_eager": ms1e, "ms_per_launch_graph_replay": ms1g,
                        "hbm_frac_per_gpu": 234 * cnt / (ms1 * 1e-3) / 1e9 / hbm_peak,
                        "note": "234 algorithmic B/env-step; 7 fp64 sin/cos pairs per step make this kernel issue-bound"}}
    env.close()
    # ---- configs[3]: reactor + SafetyWrapper bands (declarative bounds evaluated in-kernel), all-reduced counters
    n = ENVS_PER_GPU
    renv = ni.make("ChemicalReactor-v0", num_envs=n, device=f"cuda:{local}", seed=seed, env_id_offset=rank * n)
    wrapped = SafetyWrapper(renv, constraints=[
        BoundConstraint("temperature_band", 0, 280.0, 330.0, penalty=-100.0),
        BoundConstraint("pressure_band", 1, 101325.0, 400000.0, penalty=-100.0)])
    nat = wrapped.native
    nat.reset_device()
    nat.clear_stats()
    ms = timed(lambda: nat.rollout_steps_device(HORIZON, K, N.POLICY_UNIFORM), 5)       # the headline's 15 x 64 + 40 launch sequence
    allreduce_device_stats(nat)
    torch.cuda.synchronize()
    st = nat.stats_dict()
    out["reactor_safety_wrapper"] = {
        "workload": f"ChemicalReactor-v0 + SafetyWrapper(temperature 280..330 K, pressure 101325..400000 Pa, penalty -100), "
                    f"{n} envs per GPU x {world} x {HORIZON} steps, fused K=64, counters all-reduced over NCCL",
        "value": world * n * HORIZON / (ms * 1e-3), "unit": UNIT,
        "violations_per_constraint": st["violations_per_constraint"], "episodes": st["episodes"],
        "critical_shutdowns": st["critical_shutdowns"], "return_mean": st["return_sum"] / max(st["episodes"], 1)}
    renv.close()
    # ---- configs[4]: dataset writer (rank 0)
    if rank == 0:
        denv = ni.make("ChemicalReactor-v0", num_envs=1, device=f"cuda:{local}", seed=seed)
        denv.get_dataset("mixed", n_transitions=1_000_000)          # first call: allocations, page-locking of the export buffers
        dts = []
        for _ in range(3):
            t0 = time.perf_counter()
            ds = denv.get_dataset("mixed", n_transitions=1_000_000)
            dts.append(time.perf_counter() - t0)
        dt = float(np.median(dts))
        m = int(ds["rewards"].shape[0])
        out["dataset_mixed_1m"] = {
            "workload": "ChemicalReactor-v0 get_dataset('mixed') >= 1,000,000 transitions: length-probe pass + scan + write pass on the "
                        "device (D4RL layout), pinned cudaMemcpyAsync export to host numpy",
            "transitions": m, "seconds_incl_export": dt, "value": m / dt, "unit": "transitions/s", "timing": "median of 3 calls after one warm-up call",
            "terminal_rate": float(ds["terminals"].mean()), "reward_mean": float(ds["rewards"].mean())}
        denv.close()
    return out


def e2e_rollout(ni, n, local, rank, world, steps, warmup, seed, dist=None, torch=None):
    """The metric end to end through the drop-in API with HOST buffers: one bench step = one
    ``env.rollout(1000, "random", steps_per_launch=64, init_states=<pinned host array>)`` call per rank, i.e. H2D of the
    65,536 x 12 synthetic initial states, 16 fused launches, D2H of per-env returns / violation counts / episode
    counts / final observations and the stats block. Wall clock around the synchronous calls, max over ranks."""
    env = ni.make("ChemicalReactor-v0", num_envs=n, device=f"cuda:{local}", seed=seed, copy=False, env_id_offset=rank * n)
    init = env.native.pinned("init_states", (n, 12), np.float32)
    rng = np.random.default_rng(1 + rank)
    init[:] = (np.array([320, 253312.5, 50, 30, 0.5, 95, 295, 0, 0, 0, 60, 0], np.float32) +
               rng.standard_normal((n, 12)).astype(np.float32) * np.array([2, 1e4, 5, 3, 0.1, 2, 1, 0, 0, 0, 5, 0], np.float32))
    for _ in range(max(warmup, 3)):
        res = env.rollout(HORIZON, "random", steps_per_launch=K, init_states=init)
    if dist is not None:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        res = env.rollout(HORIZON, "random", steps_per_launch=K, init_states=init)
    dt = time.perf_counter() - t0
    if dist is not None:
        t = torch.tensor([dt], dtype=torch.float64, device=torch.device("cuda", local))
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    h2d = n * 12 * 4
    d2h = n * (4 + 4 + 4 + 12 * 4) + 32 * 8
    checksum = float(res["reward_sum"].astype(np.float64).sum())
    env.close()
    return {"value": world * n * HORIZON * steps / dt, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
            "ms_per_step": dt / steps * 1e3, "steps": steps,
            "api": "ni.make('ChemicalReactor-v0', num_envs=65536).rollout(1000, 'random', steps_per_launch=64, init_states=host[65536,12]) "
                   "-> host reward_sum / violations / episodes / obs / stats (C ABI: nig_rollout_host)",
            "reward_checksum_rank0": checksum}


def torch_api(torch, ni, n, local, args):
    """Secondary: the device-tensor gym API (TorchIndustrialEnv.step, zero host copies), eager and as a replayed CUDA
    graph of 50 x (torch policy -> step)."""
    env = ni.TorchIndustrialEnv("ChemicalReactor-v0", n, device=f"cuda:{local}", seed=args.seed)
    obs, _ = env.reset()
    w = torch.zeros((12, 3), device=env.device)
    w[0, 0] = -0.004

    def policy(o):
        return torch.clamp((o - 320.0) @ w, -1.0, 1.0)

    for _ in range(20):
        env.step(policy(obs))
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 500
    e0.record()
    for _ in range(reps):
        obs, r, term, trunc, info = env.step(policy(obs))
    e1.record()
    torch.cuda.synchronize()
    eager = n * reps / (e0.elapsed_time(e1) * 1e-3)
    out = {"eager": {"value": eager, "unit": UNIT, "us_per_step": e0.elapsed_time(e1) * 1e3 / reps}}
    try:
        replay = env.capture_graph(policy, 50)
        replay()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(10):
            replay()
        e1.record()
        torch.cuda.synchronize()
        out["cuda_graph"] = {"value": n * 500 / (e0.elapsed_time(e1) * 1e-3), "unit": UNIT, "us_per_step": e0.elapsed_time(e1) * 1e3 / 500}
    except Exception as ex:
        out["cuda_graph"] = {"error": repr(ex)}
    out["api"] = "ni.TorchIndustrialEnv('ChemicalReactor-v0', 65536).step(policy(obs)) with a linear torch policy; device tensors in and out"
    env.close()
    return out


def e2e_step_api(ni, n, local, args):
    """Secondary: one env.step(host actions) -> host obs / reward / terminated / truncated per call (PCIe-bound)."""
    env = ni.make("ChemicalReactor-v0", num_envs=n, device=f"cuda:{local}", seed=args.seed, copy=False)
    env.reset()
    rng = np.random.default_rng(0)
    a_buf = env.native.pinned("actions", (n, 3), np.float32)
    a_buf[:] = rng.uniform(-1, 1, (n, 3)).astype(np.float32)
    for _ in range(20):
        env.step(a_buf)
    reps = 200
    t0 = time.perf_counter()
    for _ in range(reps):
        obs, r, term, trunc, info = env.step(a_buf)
    dt = time.perf_counter() - t0
    env.close()
    return {"value": n * reps / dt, "unit": UNIT, "h2d_bytes_per_step": n * 3 * 4, "d2h_bytes_per_step": n * (12 * 4 * 2 + 4 + 1 + 1),
            "api": "env.step(actions[65536,3] host) -> obs, reward, terminated, truncated, info (one PCIe round trip per env-step)",
            "ms_per_call": dt / reps * 1e3}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--sections", default="single,e2e,cpu,configs",
                    help="extra measurements besides the headline timed region (profiling runs pass a subset)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path computed in its last step to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.sections = set(x for x in args.sections.split(",") if x)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
