"""Batch sweep of the fused x16 kernel (k23_rc_kernel<16>): `bench.py --batch B --no-e2e --no-cpu-baseline --no-secondary`
at several batch sizes, then a least-squares line kernel_us = slope * B + intercept.  The slope is the steady-state time
per image, the intercept the fixed cost of a launch (ramp and tail of the persistent grid).

usage: python tools/k23_batch_sweep.py [--root TREE] [--batches 16,24,32,64] [--steps 200] [--warmup 20]
(--root: the checkout whose bench.py is run, default this one)"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ap = argparse.ArgumentParser()
ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
ap.add_argument("--batches", default="16,24,32,64")
ap.add_argument("--steps", type=int, default=200)
ap.add_argument("--warmup", type=int, default=20)
a = ap.parse_args()

rows = []
for B in [int(b) for b in a.batches.split(",")]:
    cmd = [sys.executable, os.path.join(a.root, "bench.py"), "--batch", str(B), "--no-e2e", "--no-cpu-baseline",
           "--no-secondary", "--steps", str(a.steps), "--warmup", str(a.warmup)]
    out = subprocess.run(cmd, stdout=subprocess.PIPE, text=True, check=True).stdout
    d = [json.loads(l) for l in out.splitlines() if l.startswith("{")][-1]
    rows.append((B, d["ms_per_step"] * 1e3, d["roofline"]["kernel_us"]))
    print(f"B={B:3d}  step {rows[-1][1]:8.1f} us  k23_rc {rows[-1][2]:8.1f} us  per image {rows[-1][2] / B:6.2f} us",
          flush=True)
x = np.array([r[0] for r in rows], dtype=float)
y = np.array([r[2] for r in rows])
slope, icpt = np.polyfit(x, y, 1)
res = y - (slope * x + icpt)
print(json.dumps({"batches": x.astype(int).tolist(), "kernel_us": [round(v, 2) for v in y.tolist()],
                  "step_us": [round(r[1], 2) for r in rows], "us_per_image": round(float(slope), 3),
                  "us_per_launch": round(float(icpt), 2), "max_residual_us": round(float(np.abs(res).max()), 2)}))
