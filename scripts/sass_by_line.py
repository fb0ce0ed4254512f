#!/usr/bin/env python
"""SASS instruction count of solve_kernel per source region (code size is a first-order performance parameter: the L1.5
instruction cache holds 2048 instructions).  usage: python scripts/sass_by_line.py [libusim.so]"""
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
lib = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "robotic-ultrasound-imaging_b200", "libusim.so")
kernel = sys.argv[2] if len(sys.argv) > 2 else "solve_kernel"
with tempfile.TemporaryDirectory() as td:
    subprocess.check_call(["cuobjdump", "-xelf", "all", os.path.abspath(lib)], cwd=td, stdout=subprocess.DEVNULL)
    cub = [f for f in os.listdir(td) if f.endswith(".cubin")][0]
    sass = subprocess.run(["nvdisasm", "-g", "-c", os.path.join(td, cub)], capture_output=True, text=True).stdout
# regions of soft.cuh by line number
src = open(os.path.join(ROOT, "robotic-ultrasound-imaging_b200", "csrc", "soft.cuh")).read().splitlines()
marks = []
for i, l in enumerate(src, 1):
    m = re.search(r"auto (\w+) = \[&\]", l)
    if m:
        marks.append((i, "lambda " + m.group(1)))
    m = re.match(r"\s*// -{20,} (.*)", l)
    if m:
        marks.append((i, m.group(1)[:60]))
    m = re.match(r"__device__ __forceinline__ \S+ (\w+)\(", l)
    if m:
        marks.append((i, "fn " + m.group(1)))
    m = re.match(r"template <.*>\s*$", l)
marks.sort()


def region(line):
    name = "prologue"
    for ln, nm in marks:
        if ln <= line:
            name = nm
        else:
            break
    return name


cnt, per_line = collections.Counter(), collections.Counter()
cur_file, cur_line, in_k, total = None, 0, False, 0
# the CG loop: from the target of its back edge (a branch attributed to the K6 `for` statement) to that branch
cg_line = next(i for i, l in enumerate(src, 1) if "for (int it = -1; it < maxit; it++)" in l)
labels, back = {}, []
for l in sass.splitlines():
    if ".section" in l and ".text." in l:
        in_k = kernel in l
    if not in_k:
        continue
    m = re.search(r'//## File "(.*)", line (\d+)', l)
    if m:
        cur_file, cur_line = os.path.basename(m.group(1)), int(m.group(2))
        continue
    m = re.match(r"^\s*(\.L_x_\d+):", l)
    if m:
        labels[m.group(1)] = total
    m = re.search(r"BRA.*\(\s*(\.L_x_\d+)\s*\)", l)
    if m and cur_file == "soft.cuh" and cur_line == cg_line and m.group(1) in labels:
        back.append(total - labels[m.group(1)] + 1)
    if re.match(r"\s+/\*[0-9a-f]{4,6}\*/", l):
        total += 1
        key = region(cur_line) if cur_file == "soft.cuh" else cur_file
        cnt[key] += 1
        per_line[(cur_file, cur_line)] += 1
print(f"{kernel}: {total} SASS instructions ({total * 16 / 1024:.0f} KB)")
if back:
    print(f"CG loop (soft.cuh:{cg_line}): {max(back)} SASS instructions")
for k, v in cnt.most_common():
    print(f"{v:6d}  {k}")
print("top lines:")
for (f, ln), v in per_line.most_common(25):
    print(f"{v:6d}  {f}:{ln}  {src[ln - 1].strip()[:100] if f == 'soft.cuh' else ''}")
