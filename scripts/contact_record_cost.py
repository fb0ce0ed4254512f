#!/usr/bin/env python
"""Cost of the contact record (usim_set_contact_record) on the env step: 4096 envs in bench.py's steady-state episode mix, blocks
of steps with recording off and on alternated in one process, timed with CUDA events.

  python scripts/contact_record_cost.py [--envs 4096] [--steps 100] [--rounds 10] [--out contact_record_cost.json]

Legs: `off`; `on` (the step kernel also writes the record); `on_read` (on, plus usim_get_contact_forces into MuJoCo layouts after
every step).  Prints the GPU name and power limit with the result.
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
    ap.add_argument("--steps", type=int, default=100, help="env steps per timed block")
    ap.add_argument("--rounds", type=int, default=10, help="(off, on, on_read) blocks, alternated")
    ap.add_argument("--out", default="contact_record_cost.json", help="result file (JSON)")
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
    k = 0

    def block(leg):
        nonlocal k
        env.set_contact_record(leg != "off")
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(args.steps):
            env.step(acts[k % len(acts)])
            k += 1
            if leg == "on_read":
                env.contact_forces()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.steps

    legs = ("off", "on", "on_read")
    for leg in legs:  # warm-up of every leg
        block(leg)
    times = {leg: [] for leg in legs}
    for r in range(args.rounds):
        for leg in (legs if r % 2 == 0 else legs[::-1]):
            times[leg].append(block(leg))
    med = {leg: statistics.median(v) for leg, v in times.items()}
    res = dict(gpu=torch.cuda.get_device_name(0), nvidia_smi_name_power_limit=q.stdout.strip(), envs=args.envs, steps_per_block=args.steps,
               rounds=args.rounds, episode_mix="bench.py desync: random episode phase + one horizon of pre-roll",
               ms_per_step=times, median_ms_per_step=med,
               record_overhead_rel=med["on"] / med["off"] - 1, record_and_read_overhead_rel=med["on_read"] / med["off"] - 1)
    env.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
