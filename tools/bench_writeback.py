"""What the priority write-back costs the graphed flagship step (c51_b32, 1 M-transition shard, bench.py's HotPath
defaults): the step is captured with each write-back schedule and without the write-back (``step(update=False)``), and
the graphs are timed in alternating blocks of about 0.25 s (CUDA events, us per step).  E = step - step without
write-back is the part of the step the write-back leaves exposed.  Arms:
  planned   a0_k2b_plan after the draw + the one-CTA a0_k2b_apply under the last K4 (the default at this count)
  chunks    a0_pt_update_overlapped: the chunk K2b under the last K4 (the path above the apply's cap)
  none      no write-back
Output: one JSON object on stdout and, with --out, in that file (profiles/writeback_b200.json).

  python tools/bench_writeback.py --pairs 7 --out profiles/writeback_b200.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--workload", default="c51_b32")
ap.add_argument("--pairs", type=int, default=7, help="rounds of alternating blocks")
ap.add_argument("--block-s", type=float, default=0.25, help="device seconds per block (about)")
ap.add_argument("--out", default=None)
args = ap.parse_args()

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
torch.cuda.set_device(0)
wl = bench.WORKLOADS[args.workload]
rp, _ = bench.make_shard(wl, 1_000_000, 4, 0, torch)
hp = bench.HotPath(rp, wl, 20, 4, torch)


def capture(update, planned):
    hp._use_plan = planned and hp._use_plan_default
    rp.push_dynamic()
    for _ in range(3):
        hp.step(update=update)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        hp.step(update=update)
    hp._use_plan = hp._use_plan_default
    for _ in range(bench.SETTLE):
        g.replay()
    torch.cuda.synchronize()
    return g


arms = {"none": capture(False, False), "chunks": capture(True, False)}
if hp._use_plan_default:
    arms["planned"] = capture(True, True)


def block(g, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(20):
        g.replay()
    e0.record()
    for _ in range(steps):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / steps


steps = max(100, int(args.block_s / (block(arms["chunks"], 200) * 1e-6)))
us = {k: [] for k in arms}
for _ in range(args.pairs):
    for k, g in arms.items():
        us[k].append(round(block(g, steps), 3))
clk = subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm,power.draw", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
med = {k: float(np.median(v)) for k, v in us.items()}
out = {"gpu": gpu, "clocks_after": clk, "workload": args.workload, "transitions_per_step": hp.total, "steps_per_block": steps,
       "us_per_step": us, "median_us": {k: round(v, 3) for k, v in med.items()},
       "exposed_writeback_us": {k: round(med[k] - med["none"], 3) for k in med if k != "none"},
       "exposed_writeback_per_round_us": {k: [round(a - b, 3) for a, b in zip(us[k], us["none"])] for k in us if k != "none"}}
print(json.dumps(out))
if args.out:
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
