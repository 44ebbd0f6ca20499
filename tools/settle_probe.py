"""Why bench.py replays SETTLE untimed steps before its --warmup ones: the headline step (c51_b32, 1 M-transition
shard) is captured once, then timed in blocks of 50 replays (CUDA events, us per step) under four conditions.
Output: profiles/settle_first_replays.txt.

  python tools/settle_probe.py > profiles/settle_first_replays.txt
"""
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

smi = ["nvidia-smi", "--query-gpu=clocks.sm", "--format=csv,noheader", "-lms", "200", "-i", "0"]
print(subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip())
torch.cuda.set_device(0)
wl = bench.WORKLOADS["c51_b32"]
rp, _ = bench.make_shard(wl, 1_000_000, 4, 0, torch)
hp = bench.HotPath(rp, wl, 20, 4, torch)
rp.push_dynamic()
for _ in range(3):
    hp.step()
torch.cuda.synchronize()
g = torch.cuda.CUDAGraph()
with torch.cuda.graph(g):
    hp.step()


def blocks(n=8, warm=10, steps=50):
    for _ in range(warm):
        g.replay()
    torch.cuda.synchronize()
    out = []
    for _ in range(n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
        out.append(round(e0.elapsed_time(e1) * 1e3 / steps, 2))
    return out


print("us per step, blocks of 50 replays after 10 warm-up replays (c51_b32):")
print("right after capture          ", blocks())
print("immediately again            ", blocks())
time.sleep(1.0)
print("after 1 s idle               ", blocks())
p = subprocess.Popen(smi, stdout=subprocess.DEVNULL)
print("nvidia-smi sampler just begun", blocks())
p.terminate()
p.wait()
