"""Cost of the draw without replacement (a0_pt_sample_unique, K2a-unique) against the stratified draw with
replacement (a0_pt_sample_rng, K2a) on a 1 M-record shard, and of the graphed C51 ReplayTargetLoop step that uses it.

  sampler: CUDA events over `--launches` back-to-back launches, 20 x 32 and 20 x 512 draws, three priority vectors
           (spread |N(0,1)|-shaped, 1 % of the records at 100x, 100 records holding 90 % of the mass), with the
           rounds and candidates of a0_pt_sample_unique's stats_out.  The 8 MB tree stays in L2 between launches, as
           it does inside a training step.
  step:    one CUDA-graph replay of ReplayTargetLoop (C51, L = 20 batches) at B = 32 and B = 512: with replacement
           and the default gather waves, with replacement and one plain gather launch, and without replacement.

Run on the GPU: python tools/bench_sample_unique.py [--out FILE]; prints one JSON line per row and the card's name
and power limit, and with --out also writes everything to FILE (profiles/sample_unique_b200.json is such a file)."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import bench  # noqa: E402
from agent0_b200 import _lib  # noqa: E402
from agent0_b200.config import make_config  # noqa: E402
from agent0_b200.hotloop import ReplayTargetLoop  # noqa: E402
from agent0_b200.replay import ReplayDataset  # noqa: E402

N, E, A, L = 1_000_000, 16, 4, 20


def events_us(fn, n):
    for _ in range(10):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) * 1e3 / n


def set_vector(rp, kind, live, saved):
    dev = rp.device
    g = torch.Generator(device=dev).manual_seed(9)
    if kind == "spread":
        v = saved
    else:
        v = torch.ones(live.numel(), device=dev)
        heavy = torch.randperm(live.numel(), device=dev, generator=g)[:live.numel() // 100]
        v[heavy] = 100.0
        if kind == "extreme_100_records_hold_90pct":
            v = torch.ones(live.numel(), device=dev)
            v[heavy[:100]] = 0.9 / 0.1 * float(live.numel() - 100) / 100.0
    for lo in range(0, live.numel(), 1 << 20):
        rp.set_priorities(live[lo:lo + (1 << 20)], v[lo:lo + (1 << 20)])
    torch.cuda.synchronize()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="JSON file for the card name and every row")
    ap.add_argument("--launches", type=int, default=500)
    ap.add_argument("--replays", type=int, default=300)
    args = ap.parse_args()
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    print(json.dumps({"card": card}), flush=True)
    lib = _lib.load()
    rows = []
    cfg = make_config("c51", per=True, n_step=3, batch_size=32, replay_size=N, double_q=True, dueling=True, num_envs=E,
                      action_dim=A)
    rp = ReplayDataset(cfg, native_nstep=True)
    bench.fill_shard(rp, N, E, 1234, torch)
    dev = rp.device
    leaves = rp.priority.leaves()
    live = torch.nonzero(leaves > 0).squeeze(1)
    g = torch.Generator(device=dev).manual_seed(5)
    spread = (torch.randn(live.numel(), device=dev, generator=g).abs() + 0.01).sqrt()
    st = _lib.stream_ptr(dev)
    top = float(rp.top)
    for kind in ("spread", "peaked_1pct_at_100x", "extreme_100_records_hold_90pct"):
        set_vector(rp, kind, live, spread)
        for B in (32, 512):
            T = L * B
            idx = torch.empty(T, dtype=torch.int64, device=dev)
            prio, w = torch.empty(T, device=dev), torch.empty(T, device=dev)
            stats = torch.empty((L, 2), dtype=torch.int32, device=dev)
            rng = lambda: lib.a0_pt_sample_rng(rp.h, 7, -1, T, B, top, 0.4, 0.0, 0, idx.data_ptr(), prio.data_ptr(),
                                               w.data_ptr(), None, st)
            uniq = lambda: lib.a0_pt_sample_unique(rp.h, 7, -1, T, B, top, 0.4, 0.0, 0, idx.data_ptr(), prio.data_ptr(),
                                                   w.data_ptr(), stats.data_ptr(), st)
            _lib.check(uniq(), "a0_pt_sample_unique")
            torch.cuda.synchronize()
            s = stats.float()
            dups = sum(B - int(torch.unique(idx.view(L, B)[k]).numel()) for k in range(L))
            row = {"kind": "sampler", "priorities": kind, "draw": f"{L}x{B}",
                   "a0_pt_sample_rng_us": round(events_us(rng, args.launches), 2),
                   "a0_pt_sample_unique_us": round(events_us(uniq, args.launches), 2),
                   "unique_rounds_mean": round(float(s[:, 0].mean()), 3), "unique_rounds_max": int(s[:, 0].max()),
                   "unique_candidates_mean": round(float(s[:, 1].mean()), 1), "unique_duplicates": dups}
            print(json.dumps(row), flush=True)
            rows.append(row)
    set_vector(rp, "spread", live, spread)
    for B in (32, 512):
        o = bench.net_outputs("c51", L * B, A, torch, dev)
        for mode, kw in (("with_replacement_waves", {}), ("with_replacement_no_overlap", {"overlap_sample_gather": False}),
                         ("without_replacement", {"replacement": False})):
            loop = ReplayTargetLoop(rp, "c51", B, L, A, o, n_step=3, rng_seed=3, **kw)
            loop.capture()
            rp.push_dynamic()
            us = events_us(loop.graph.replay, args.replays)
            row = {"kind": "graphed_c51_step", "B": B, "L": L, "mode": mode, "step_us": round(us, 1),
                   "per_update_us": round(us / L, 2)}
            print(json.dumps(row), flush=True)
            rows.append(row)
            del loop
            torch.cuda.synchronize()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump({"card": card, "shard_records": N, "rows": rows}, f, indent=1)
            f.write("\n")


if __name__ == "__main__":
    main()
