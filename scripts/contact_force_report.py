#!/usr/bin/env python
"""Measured fp32-vs-float64 agreement of the contact record (usim_get_contact_forces) with the oracle's contacts: the maxima the
tolerances of tests/test_contact_forces.py are derived from.

  python scripts/contact_force_report.py [--out contact_force_parity.json]

Runs tests/contact_util.contact_parity (the test's own comparison) for the soft and the rigid scene.  force_rel: per env-step, the
largest |df_c| (frame-coordinate force on geom2) over max(1 N, sum_c f_n,c); pos / frame: largest absolute entry difference.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from contact_util import contact_parity  # noqa: E402


def gpu_info():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return dict(gpu=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="contact_force_parity.json", help="result file (JSON)")
    args = ap.parse_args()
    from oracle import oracle as O
    O.lib()
    res = dict(gpu_info(), metric="force_rel: max over env-steps of max_c |df_c| / max(1 N, sum_c f_n,c); pos, frame: max |d|")
    for name, soft in (("soft_box_tracking", True), ("rigid_fixed_press", False)):
        res[name] = contact_parity(O, soft)
        print(name, json.dumps(res[name]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
