"""Measure the solve-on-identical-inputs maxima that tests/test_solve_identical_inputs.py bounds (tests/solve_util.py does the
comparing); writes profiles/solve_parity.json, or --out.

    python scripts/solve_parity_report.py [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import solve_util as su  # noqa: E402
from oracle import oracle as O  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "solve_parity.json"))
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    # stats of every group: maxima of the metrics (tests/solve_util.stats); knobs: cap monotonicity, line searches, tolerance and
    # rebuild settings (solve_util.knob_stats); limits: the joint-limit cases of both robots
    res = dict(gpu=gpu, groups={}, knobs={}, limits={}, seconds={})
    for name in ("soft", "rigid", "cylinder", "ur5e"):
        t0 = time.time()
        params, cc = su.scene(name)
        knobs = list(su.KNOBS) if name in ("soft", "rigid") else ["default"]
        by = su.run(O, params, cc, su.trajectory_batches(O, name), knobs)
        res["groups"][name] = su.stats([r for recs in by.values() for r in recs])
        res["groups"][name]["default_capped"] = su.stats(by["default"])["capped"]
        if name in ("soft", "rigid"):
            res["knobs"][name] = su.knob_stats(by)
        res["seconds"][name] = round(time.time() - t0)
        print(name, json.dumps(res["groups"][name]), json.dumps(res["knobs"].get(name)), flush=True)
    for robot in ("panda", "ur5e"):
        t0 = time.time()
        lr = su.limit_records(O, robot)
        res["groups"][f"limit_{robot}_soft"] = su.stats(lr["soft"])
        res["groups"][f"limit_{robot}_rigid"] = su.stats([r for recs in lr["rigid"].values() for r in recs])
        res["limits"][robot] = dict(cap_increase=su.cap_increase(lr["rigid"]), **{
            k: v for k, v in su.knob_stats(lr["rigid"]).items() if k.startswith("line_search")},
            soft_cases=len(lr["soft"]), rigid_cases=len(lr["rigid"]["default"]), soft_nlim=sorted({r["nlim"] for r in lr["soft"]}),
            rigid_ncon_zero=sum(r["ncon"] == 0 for r in lr["rigid"]["default"]))
        res["seconds"]["limits_" + robot] = round(time.time() - t0)
        print(robot, json.dumps(res["groups"][f"limit_{robot}_soft"]), json.dumps(res["groups"][f"limit_{robot}_rigid"]),
              json.dumps(res["limits"][robot]), flush=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
