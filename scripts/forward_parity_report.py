"""Measure the forward-pass-on-identical-inputs maxima that tests/test_forward.py bounds (tests/forward_util.py does the comparing);
writes profiles/forward_parity.json, or --out.

    python scripts/forward_parity_report.py [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import forward_util as fu  # noqa: E402
from oracle import oracle as O  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "forward_parity.json"))
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    # per scene and torque kind: maxima of the metrics (forward_util.stats); "scenes": both torque kinds together
    res = dict(gpu=gpu, groups={}, scenes={}, seconds={})
    for name in fu.SCENES:
        t0 = time.time()
        both = []
        for kind in fu.CTRLS:
            recs = fu.run(O, name, kind)
            res["groups"][f"{name}_{kind}"] = fu.stats(recs)
            both += recs
            print(name, kind, json.dumps(res["groups"][f"{name}_{kind}"]), flush=True)
        res["scenes"][name] = fu.stats(both)
        res["seconds"][name] = round(time.time() - t0)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["scenes"], indent=1))


if __name__ == "__main__":
    main()
