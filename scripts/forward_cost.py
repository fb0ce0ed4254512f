#!/usr/bin/env python
"""Cost of a forward pass (usim_forward) next to the env step: 4096 envs in bench.py's steady-state episode mix, blocks of steps and
blocks of forward passes alternated in one process, timed with CUDA events.

  python scripts/forward_cost.py [--envs 4096] [--calls 100] [--rounds 10] [--out profiles/forward_cost.json]

Legs: `step` (one env step); `forward` (forward() with zero torques, observation into env.obs); `forward_ctrl_qacc` (forward with a
torque row and the qacc output).  The forward passes run at the state the last step left, so they solve the same problems a step
of that state would, from its warm start.  Prints the GPU name and power limit with the result.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--calls", type=int, default=100, help="calls per timed block")
    ap.add_argument("--rounds", type=int, default=10, help="(step, forward, forward_ctrl_qacc) blocks, alternated")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "forward_cost.json"), help="result file (JSON)")
    args = ap.parse_args()
    import torch

    import bench
    from rui_b200.env import BatchedUltrasound

    dev = torch.device("cuda:0")
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    env = BatchedUltrasound(args.envs, device=0, seed=bench.SEED, **bench.ENV_OPTS)
    gen = torch.Generator(device=dev).manual_seed(bench.SEED)
    acts = [torch.rand(args.envs, env.action_dim, device=dev, generator=gen) for _ in range(64)]
    bench.desync(env, acts, gen, -1)
    rng = torch.as_tensor(env.model.g_ctrl_range, dtype=torch.float32, device=dev)
    ctrl = (torch.rand(args.envs, 7, device=dev, generator=gen) * 2 - 1) * rng
    k = 0

    def block(leg):
        nonlocal k
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(args.calls):
            if leg == "step":
                env.step(acts[k % len(acts)])
                k += 1
            elif leg == "forward":
                env.forward()
            else:
                env.forward(ctrl=ctrl, qacc=True)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.calls

    legs = ("step", "forward", "forward_ctrl_qacc")
    for leg in legs:  # warm-up of every leg
        block(leg)
    times = {leg: [] for leg in legs}
    for r in range(args.rounds):
        for leg in (legs if r % 2 == 0 else legs[::-1]):
            times[leg].append(block(leg))
    med = {leg: statistics.median(v) for leg, v in times.items()}
    res = dict(gpu=torch.cuda.get_device_name(0), nvidia_smi_name_power_limit=q.stdout.strip(), envs=args.envs, calls_per_block=args.calls,
               rounds=args.rounds, episode_mix="bench.py desync: random episode phase + one horizon of pre-roll",
               ms_per_call=times, median_ms_per_call=med, spread_ms={leg: [min(v), max(v)] for leg, v in times.items()},
               forward_over_step=med["forward"] / med["step"])
    env.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
