#!/usr/bin/env python
"""Benchmark of the Ultrasound env step (BASELINE.json metric: env-steps/s, soft-torso sweep task).

  python bench.py --gpus N --steps K --warmup W            # CUDA path (this repo)
  python bench.py --impl reference --gpus N --steps K ...  # CPU arm: float64 oracle port on the host cores

One "step" = one control step (= one 0.002 s physics step) of EVERY env of the batch, random actions,
auto-reset on.  N=1: BASELINE config 3 (4096 envs on one B200).  N>1: config 4 (65536 envs split evenly
over the ranks, one process per GPU, no data-path collective; envs never interact).
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ALG_BYTES_PER_ENV_STEP = 7008  # SURVEY.md §8(d): fp32 state read+written once per step, soft config
RL_CONTROLLER = dict(  # src/rl_config.yaml:33-51 of the reference
    type="OSC_POSE", input_max=1, input_min=-1, output_max=[0.05, 0.05, 0.05, 0.5, 0.5, 0.5],
    output_min=[-0.05, -0.05, -0.05, -0.5, -0.5, -0.5], kp=300, damping_ratio=1, impedance_mode="tracking",
    kp_limits=[0, 500], kp_input_max=1, kp_input_min=0, damping_ratio_limits=[0, 2], position_limits=None,
    orientation_limits=None, uncouple_pos_ori=True, control_delta=True, interpolation=None, ramp_ratio=0.2)
ENV_OPTS = dict(controller_configs=RL_CONTROLLER, control_freq=500, horizon=1000, early_termination=False,
                torso_solref_randomization=True, initial_probe_pos_randomization=True)
SEED = 3  # rl_config.yaml:1


def _ncu_capture():
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None
    with open(p) as f:
        return json.load(f)


def ncu_traffic(envs_per_gpu):
    """dram bytes per launch of the dominant kernel from the committed ncu capture (scaled to this launch's env count)."""
    t = _ncu_capture()
    return None if t is None else t["dram_bytes_per_launch"] * envs_per_gpu / t["envs_per_launch"]


def issue_slots(envs_per_gpu, kernel_ms, sm_mhz, mean_iters, n_sm=148):
    """The bound that actually applies (DESIGN.md §4/§6): warp instructions issued per second against 4 schedulers x SMs x clock.
    Instructions per launch = the committed ncu capture's count, scaled to this launch's env count and to the LIVE solver work:
    the loop share of the instructions (80 %, profiles/r02_ncu_source_regions.txt) scales with the CG iterations per env-step
    counted by the kernel in this very run (diag[20]); the time is measured live."""
    t = _ncu_capture()
    if t is None or "warp_instructions_per_launch" not in t or not sm_mhz:
        return None
    loop = t.get("loop_share_of_instructions", 0.8)
    it0 = t.get("mean_solver_iters_of_capture") or mean_iters
    inst = t["warp_instructions_per_launch"] * envs_per_gpu / t["envs_per_launch"] * ((1 - loop) + loop * mean_iters / it0)
    achieved = inst / (kernel_ms * 1e-3) / 1e9
    peak = 4 * n_sm * sm_mhz * 1e6 / 1e9
    return {"bound": "fp32 issue slots (secondary, informative)", "achieved": achieved, "peak": peak, "unit": "G warp-instr/s",
            "frac": achieved / peak, "live_mean_cg_iterations": mean_iters,
            "source": "smsp__inst_executed.sum of the committed capture (profiles/traffic.json) scaled by the live CG iteration count, over the live kernel time"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons of one GPU while the timed region runs."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "sw_power_cap": 0x4,
                 "hw_power_brake_slowdown": 0x80}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.05)

    def result(self):
        self.stop_flag = True
        if self.nv is None or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def cpu_baseline(threads: int, steps: int, repeats: int = 3):
    """Float64 oracle port on the host cores: `threads` envs, one per thread, `steps` env steps each."""
    from oracle import oracle as O
    from rui_b200.abi import PackedModel, make_config
    from rui_b200.model import build_model

    pk = PackedModel(build_model())
    envs = []
    for i in range(threads):
        cfg = make_config(1, RL_CONTROLLER, seed=SEED, **{k: v for k, v in ENV_OPTS.items() if k != "controller_configs"})
        e = O.OracleEnv(pk, cfg, i)
        e.set_forward_repeats(repeats)  # the reference runs mj_forward three times per step (SURVEY §3.2)
        e.reset()
        envs.append(e)
    rng = np.random.default_rng(SEED)
    acts = rng.uniform(0, 1, size=(steps, threads, 6))
    O.rollout(envs, acts[:2], auto_reset=True, threads=threads)  # warm caches
    t0 = time.perf_counter()
    n, _ = O.rollout(envs, acts, auto_reset=True, threads=threads)
    dt = time.perf_counter() - t0
    return n / dt, dt, envs, pk


def run_reference(args):
    """--impl reference: the reference's CPU path cannot be installed here (MuJoCo 2.0 binary + un-vendored forks,
    SURVEY §8c), so the float64 oracle port is timed on all host cores, doing the reference's three forward passes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O
    threads = os.cpu_count() or 1
    rate0, _, envs, _ = cpu_baseline(threads, 3)
    rng = np.random.default_rng(SEED + 1)
    per_step = max(1, int(min(20.0, 120.0 / max(args.steps + args.warmup, 1)) * rate0 / threads))  # env steps per thread per bench step
    acts = rng.uniform(0, 1, size=(per_step, threads, 6))
    for _ in range(args.warmup):
        O.rollout(envs, acts, auto_reset=True, threads=threads)
    t0 = time.perf_counter()
    tot = 0
    for _ in range(args.steps):
        n, _ = O.rollout(envs, acts, auto_reset=True, threads=threads)
        tot += n
    dt = time.perf_counter() - t0
    val = tot / dt
    # BASELINE config 1 literally: ONE env on one host core (the shape the reference's Ultrasound env has inside each SubprocVecEnv worker)
    one = envs[:1]
    a1 = rng.uniform(0, 1, size=(max(40, int(3.0 * rate0 / threads)), 1, 6))
    t1 = time.perf_counter()
    n1, _ = O.rollout(one, a1, auto_reset=True, threads=1)
    single = n1 / (time.perf_counter() - t1)
    line = {
        "impl": "reference", "metric": "ultrasound env-steps/sec", "value": val, "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "soft-torso sweep task, rl_config.yaml controller, random actions U[0,1]^6, auto-reset",
                   "envs": threads, "env_steps_per_bench_step": per_step * threads},
        "cpu_baseline": {"value": val, "unit": "env-steps/s", "cores": threads, "kind": "port",
                         "sample": f"{threads} envs x {per_step} steps per bench step, 3 forward passes per step as in the reference"},
        "e2e": {"value": val, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "config1_single_env": {"value": single, "unit": "env-steps/s", "cores": 1, "sample": f"1 env x {a1.shape[0]} steps",
                               "note": "BASELINE config 1: single env, OSC_POSE, random actions, one host core"},
        "note": "restated-reference CPU baseline (mujoco-py unavailable): a float64 port of the published algorithms, NOT mujoco-py; "
                "artifact-derived historical figure of the reference itself: 385.5 env-steps/s on 64 workers (6 per worker, PPO updates and hard resets included)",
    }
    print(json.dumps(line), flush=True)


def desync(env, acts, gen, preroll):
    """Steady-state episode mix, independent of --steps / --warmup: every env gets a uniformly random episode phase
    (MujocoEnv.timestep through usim_set_state), then `preroll` untimed steps (default: one full horizon) are run, so that
    every env has been through a reset at a uniformly distributed time: the timed window sees resets staggered at ~N / horizon
    per step and post-reset transients in their natural proportion, as a long RL run does -- not the lock-step start."""
    import torch

    from rui_b200 import abi
    env.reset()
    q, v, w, t = env.get_state()
    t[:, abi.TS_TIMESTEP] = torch.randint(0, env.horizon, (env.num_envs,), device=t.device, generator=gen).float()
    env.set_state(task=t)
    n = env.horizon if preroll < 0 else preroll
    for i in range(n):
        env.step(acts[i % len(acts)])
    torch.cuda.synchronize()
    return n


DUMP_NAMES = ("obs", "reward", "done", "terminal_obs")  # what BatchedUltrasound.step returns, in that order
DUMP_MAX_BYTES = 64 << 20


def dump_outputs(dirname, outputs, world, rank):
    """Write what the last timed step returned as float32 DIR/<name>.npy (rows of all ranks, in global env order), so that two
    builds can be compared output for output.  Above DUMP_MAX_BYTES a fixed, seeded sample of env rows is written, with its global
    env ids in DIR/env_index.npy."""
    import torch
    import torch.distributed as dist

    arrays = {}
    for name, t in zip(DUMP_NAMES, outputs):
        t = t.float()
        if world > 1:
            parts = [torch.empty_like(t) for _ in range(world)]
            dist.all_gather(parts, t)
            t = torch.cat(parts)
        arrays[name] = t.cpu().numpy()
    if rank != 0:
        return
    n = len(arrays["obs"])
    row_bytes = sum(a[:1].nbytes for a in arrays.values())
    if n * row_bytes > DUMP_MAX_BYTES:
        k = (DUMP_MAX_BYTES - 4096) // (row_bytes + 8)  # (4 KiB: the .npy headers)
        rows = np.sort(np.random.default_rng(SEED).choice(n, size=k, replace=False))
        arrays = {name: a[rows] for name, a in arrays.items()}
        arrays["env_index"] = rows.astype(np.float64)
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


def run_cuda(args):
    import torch
    import torch.distributed as dist

    from rui_b200.env import BatchedUltrasound

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    if args.envs:
        per_gpu = args.envs
    else:
        per_gpu = 4096 if world == 1 else 65536 // world
    env = BatchedUltrasound(per_gpu, device=dev, seed=SEED, env_id_offset=rank * per_gpu, solver_iterations=args.iters, precond_rebuilds=args.rebuilds, **({"solver_tolerance": args.tol} if args.tol else {}), **ENV_OPTS)
    gen = torch.Generator(device=dev)
    gen.manual_seed(SEED + rank)
    nact = 8
    acts = [torch.rand(per_gpu, env.action_dim, device=dev, generator=gen) for _ in range(nact)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev) if not args.no_flush else None
    preroll = desync(env, acts, gen, args.preroll)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident throughput
    for i in range(args.warmup):
        env.step(acts[i % nact])
    env.set_timing(True)  # CUDA events around the dominant kernel (opt-in: off in production)
    env.kernel_time(reset=True)
    sampler = ClockSampler(local)
    sampler.start()
    l0 = env.launch_count
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    t_wall = time.perf_counter()
    for i in range(args.steps):
        if flush is not None:
            flush.zero_()
        evs[i][0].record()
        last = env.step(acts[i % nact])
        evs[i][1].record()
    barrier()
    t_wall = time.perf_counter() - t_wall
    launches = env.launch_count - l0
    clocks = sampler.result()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last, world, rank)
    ms = sum(a.elapsed_time(b) for a, b in evs)
    kms, kn = env.kernel_time(reset=True)
    env.set_timing(False)
    diag = env.diag()
    mean_ncon, mean_iters = float(diag[:, 22].mean()), float(diag[:, 20].mean())
    mean_rebuilds, mean_ls = float(diag[:, 24].mean()), float(diag[:, 25].mean())

    # ---------------- end to end through the host-buffer C-ABI call (H2D actions, D2H obs/reward/done inside)
    acts_h = [a.cpu().pin_memory().numpy() for a in acts]  # pinned host inputs, pinned host results (env.step_host)
    for i in range(min(args.warmup, 3)):
        env.step_host(acts_h[i % nact])
    barrier()
    t0 = time.perf_counter()
    for i in range(args.steps):
        env.step_host(acts_h[i % nact])
    barrier()
    e2e_s = time.perf_counter() - t0

    t = torch.tensor([ms, e2e_s * 1e3, kms / max(kn, 1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max, e2e_ms_max, kernel_ms = [float(x) for x in t.tolist()]
    total_envs = per_gpu * world
    value = total_envs * args.steps / (ms_max * 1e-3)
    e2e = total_envs * args.steps / (e2e_ms_max * 1e-3)

    # N > 1 (config 4: 65536 envs split over the ranks): the honest denominator of a scaling efficiency is ONE GPU running all
    # 65536 envs, not the 4096-env N=1 line (a smaller batch per GPU has a longer launch tail).  Rank 0 measures it here, with
    # the same pre-roll and timing, while the other ranks wait.
    strong_ref = None
    if world > 1 and not args.no_strong_ref:
        if rank == 0:
            env.close()
            big = BatchedUltrasound(total_envs, device=dev, seed=SEED, env_id_offset=0, solver_iterations=args.iters,
                                    precond_rebuilds=args.rebuilds, **({"solver_tolerance": args.tol} if args.tol else {}), **ENV_OPTS)
            bacts = [torch.rand(total_envs, big.action_dim, device=dev, generator=gen) for _ in range(nact)]
            desync(big, bacts, gen, args.preroll)
            bev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
            for i in range(args.steps):
                if flush is not None:
                    flush.zero_()
                bev[i][0].record()
                big.step(bacts[i % nact])
                bev[i][1].record()
            torch.cuda.synchronize()
            bms = sum(a.elapsed_time(b) for a, b in bev)
            strong_ref = {"n_gpus": 1, "envs": total_envs, "value": total_envs * args.steps / (bms * 1e-3), "unit": "env-steps/s",
                          "ms_per_step": bms / args.steps, "note": "same workload on ONE GPU (rank 0), measured in this run"}
            big.close()
        barrier()

    # BASELINE config 5 in the same run (all ranks: the gradient all-reduce is an NCCL collective), so that the PPO figure is in the
    # driver's record too; a few seconds
    ppo = None
    if not args.no_ppo:
        env.close()  # (idempotent; rank 0 may have closed it for the strong_ref measurement)
        ppo = measure_ppo(args, world, rank, local, args.ppo_iters, 3)

    if rank == 0:
        peak, which = peaks()
        achieved = per_gpu * ALG_BYTES_PER_ENV_STEP / (kernel_ms * 1e-3) / 1e9
        line = {
            "metric": "ultrasound env-steps/sec", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True,
            "scaling": "weak" if world == 1 else "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": ("BASELINE config 3: soft-torso sweep task, 4096 envs on 1 B200" if world == 1 and not args.envs else
                                    f"BASELINE config 4: soft-torso sweep task, {total_envs} envs over {world} GPU(s)"),
                       "envs_total": total_envs, "envs_per_gpu": per_gpu, "controller": "OSC_POSE tracking (rl_config.yaml)",
                       "actions": "U[0,1]^6 (torch.Generator seed 3)", "auto_reset": True,
                       "early_termination": ENV_OPTS["early_termination"],
                       "episode_phase": f"uniformly random per env + {preroll} untimed pre-roll steps (steady-state mix of resets and "
                                        "post-reset transients; independent of --steps/--warmup)",
                       "solver": f"PCG cap {args.iters}, relative gradient tolerance {args.tol or 3e-5:g}", "mean_ncon": mean_ncon, "mean_solver_iters": mean_iters,
                       "mean_precond_rebuilds": mean_rebuilds, "mean_line_search_evals": mean_ls,
                       "l2": "state (~37 MB at 4096 envs) is smaller than L2; 256 MiB memset between steps, outside the per-step events"
                             if flush is not None else "not flushed"},
            "clocks": clocks,
            "e2e": {"value": e2e, "unit": "env-steps/s", "h2d_bytes_per_step": per_gpu * env.action_dim * 4,
                    "d2h_bytes_per_step": per_gpu * (19 * 4 + 4 + 1),
                    "note": "usim_step_host with page-locked host buffers: actions host->device by cudaMemcpyAsync; obs + reward + done "
                            "rows (and the terminal rows of the envs that finished in the step) device->host as posted writes of the step "
                            "kernel into the mapped result buffers, inside the timed region; stream synchronised every step.  "
                            "early_termination off as in the device-resident line (rl_config.yaml:53 trains with it on: --early-termination)"},
            "gpu_launches": int(launches),
            "wall_s_timed_region": t_wall,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": args.traffic if args.traffic is not None else ncu_traffic(per_gpu), "kernel": "solve_kernel", "kernel_ms": kernel_ms, "peak_source": which,
                         "note": "algorithmic bytes 7008 B/env-step (SURVEY 8d); the step is FP32-issue/latency bound, not HBM bound"},
        }
        if strong_ref is not None:
            line["strong_ref"] = strong_ref
        if ppo is not None:
            line["ppo"] = {k: v for k, v in ppo.items() if k != "clocks"}
        iss = issue_slots(per_gpu, kernel_ms, clocks.get("sm_mhz"), mean_iters)
        if iss is not None:
            line["issue_slots"] = iss
        if world == 1 and not args.no_cpu:
            threads = os.cpu_count() or 1
            if args.cpu_steps <= 0:  # bounded sample: 10-20 s of CPU work, sized from a short calibration run
                r0, _, _, _ = cpu_baseline(threads, 4)
                args.cpu_steps = int(min(max(22.0 * r0 / threads, 20), 5000))
            rate, dt, _, _ = cpu_baseline(threads, args.cpu_steps)
            line["cpu_baseline"] = {"value": rate, "unit": "env-steps/s", "cores": threads, "kind": "port",
                                    "sample": f"{threads} envs x {args.cpu_steps} steps of the same workload, float64 oracle with the "
                                              f"reference's 3 forward passes per step ({dt:.1f} s)"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def measure_ppo(args, world, rank, local, steps, warmup):
    """BASELINE config 5 -- PPO training from rl_config.yaml hyper-parameters on GPU-batched rollouts, one process per GPU, envs
    sharded over the ranks, gradients averaged by one flat NCCL all-reduce per minibatch.  One "step" here = one PPO iteration = a
    rollout of n_steps control steps of every env + n_epochs x minibatches optimiser steps.  Returns the result dict on rank 0."""
    import torch
    import torch.distributed as dist

    from rui_b200.env import BatchedUltrasound
    from rui_b200.ppo import PPO

    dev = torch.device(f"cuda:{local}")
    per_gpu = args.ppo_envs  # config 5 at 8 GPUs: 65536 envs
    opts = dict(ENV_OPTS, early_termination=True)  # rl_config.yaml:53
    env = BatchedUltrasound(per_gpu, device=dev, seed=SEED, env_id_offset=rank * per_gpu, **opts)
    n_steps = args.n_steps
    model = PPO(env, n_steps=n_steps, seed=SEED, net_arch=[dict(pi=[256, 128], vf=[256, 128])])  # rl_config.yaml:13-16
    model.profile_allreduce = world > 1

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    model._setup()
    for _ in range(max(warmup, 3)):  # includes the CUDA-graph capture of the minibatch step
        model.train(model.collect_rollouts())
    model.allreduce_ms()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = env.launch_count
    e0, e1, er = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), []
    barrier()
    e0.record()
    for _ in range(steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        batch = model.collect_rollouts()
        b.record()
        er.append((a, b))
        model.train(batch)
    e1.record()
    barrier()
    clocks = sampler.result()
    ms = e0.elapsed_time(e1)
    rollout_ms = sum(a.elapsed_time(b) for a, b in er)
    ar_ms, ar_n = model.allreduce_ms()
    t = torch.tensor([ms, ar_ms, rollout_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max, ar_max, ro_max = [float(x) for x in t.tolist()]
    total = per_gpu * world * n_steps * steps
    launches = int(env.launch_count - l0)
    stats = dict(model.last_stats)
    nmb = (per_gpu * n_steps) // model.batch_size
    res = {
        "value": total / (ms_max * 1e-3), "unit": "env-steps/s", "n_gpus": world, "iterations": steps, "ms_per_iteration": ms_max / steps,
        "rollout_ms_per_iteration": ro_max / steps, "update_ms_per_iteration": (ms_max - ro_max) / steps,
        "allreduce_ms_per_iteration": ar_max / steps, "allreduces_per_iteration": ar_n / max(steps, 1),
        "allreduce_bytes": 4 * sum(p.numel() for p in model.policy.parameters()),
        "config": {"workload": f"BASELINE config 5: PPO training (rl_config.yaml hyper-parameters) on {per_gpu * world} GPU-batched envs, "
                               f"{world} GPU(s), NCCL gradient all-reduce",
                   "envs_total": per_gpu * world, "envs_per_gpu": per_gpu, "n_steps": n_steps,
                   "n_steps_note": "the reference's 2048 x 64 envs; 2048 x 65536 would exceed total_timesteps (SURVEY 8d cfg 5)",
                   "n_epochs": model.n_epochs, "minibatches_per_epoch": nmb, "batch_size_per_gpu": model.batch_size,
                   "iteration": "rollout (n_steps control steps of every env) + update", "early_termination": True,
                   "policy": "MlpPolicy pi/vf [256,128] (76,941 parameters), random init"},
        "step_reward_mean": stats.get("step_reward_mean"), "ep_len_mean": stats.get("ep_len_mean"), "gpu_launches": launches, "clocks": clocks,
    }
    env.close()
    return res


def run_ppo(args):
    """--workload ppo: the config-5 measurement as the line's own value."""
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    torch.cuda.set_device(local)
    args.ppo_envs = args.envs or args.ppo_envs
    r = measure_ppo(args, world, rank, local, args.steps, args.warmup)
    if rank == 0:
        line = {
            "metric": "ultrasound env-steps/sec", "value": r["value"], "unit": "env-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": r["ms_per_iteration"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(r["config"], bench_step="one PPO iteration", l2="not flushed (the update streams ~100 MB of rollout buffers per epoch)"),
            "clocks": r["clocks"], "gpu_launches": r["gpu_launches"],
            "ppo": {k: r[k] for k in ("rollout_ms_per_iteration", "update_ms_per_iteration", "allreduce_ms_per_iteration",
                                      "allreduces_per_iteration", "allreduce_bytes", "step_reward_mean", "ep_len_mean")},
            "e2e": {"value": r["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                    "note": "training keeps observations, actions and rewards on the device: there is no host hop in this workload"},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--workload", default="env", choices=["env", "ppo"], help="env: the env step (configs 3/4, default); ppo: config 5")
    ap.add_argument("--n-steps", type=int, default=32, help="PPO: rollout length per iteration")
    ap.add_argument("--ppo-envs", type=int, default=8192, help="PPO: envs per GPU (config 5: 65536 over 8 GPUs)")
    ap.add_argument("--ppo-iters", type=int, default=3, help="PPO iterations timed at the end of the default run (config 5 sub-record)")
    ap.add_argument("--no-ppo", action="store_true", help="skip the config-5 PPO sub-measurement of the default run")
    ap.add_argument("--envs", type=int, default=0, help="envs per GPU (default: BASELINE configs)")
    ap.add_argument("--iters", type=int, default=40, help="solver iteration cap")
    ap.add_argument("--rebuilds", type=int, default=0, help="preconditioner rebuilds allowed per solve (0: library default)")
    ap.add_argument("--tol", type=float, default=0.0, help="device solver tolerance (0: library default 3e-5)")
    ap.add_argument("--preroll", type=int, default=-1, help="untimed steps after randomising the episode phases (-1: one horizon)")
    ap.add_argument("--early-termination", action="store_true", help="rl_config.yaml:53 (episodes then last tens of steps under random actions)")
    ap.add_argument("--no-flush", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-strong-ref", action="store_true", help="N>1: skip the 1-GPU x all-envs reference measurement on rank 0")
    ap.add_argument("--cpu-steps", type=int, default=0, help="env steps per host thread of the cpu_baseline sample (0: ~15 s of CPU work)")
    ap.add_argument("--traffic", type=float, default=None, help="dram bytes per launch of the dominant kernel from an ncu capture")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="env workload: write what the last timed step returned (obs, reward, done, terminal_obs) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "cuda" or args.workload != "env"):
        ap.error("--dump-outputs applies to the CUDA env-step workload")
    if args.early_termination:
        ENV_OPTS["early_termination"] = True
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "ppo":
        run_ppo(args)
    else:
        run_cuda(args)


if __name__ == "__main__":
    main()
