"""Phases of merging shard checkpoints into a shard of another capacity (a0_ckpt_merge, ReplayDataset.load_merged)
against the exact resume (a0_ckpt_load).

C51 shards of --records records (n = 3, native ingest) are filled with bench_checkpoint's Atari-like frames and saved
to a temporary directory.  Cases: ``load`` into the same shape; ``load_merged`` of the one file into the same shape,
into a shard of half and of twice the records; two files merged into one shard of twice the records.  For each: total
time, validation, host merge plan, decode + place (CUDA events), records + leaves, bytes decoded and placed, and the
wall time around the call (ending in a device synchronise).  Every case runs once to warm up and is timed on the
second run.  Writes one JSON object with the card's name and power limit to --out."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from agent0_b200.config import make_config  # noqa: E402
from agent0_b200.replay import ReplayDataset  # noqa: E402
from bench_checkpoint import atari_fill  # noqa: E402


def _shard(records):
    cfg = make_config("c51", per=True, n_step=3, batch_size=32, replay_size=records, double_q=True, dueling=True)
    return ReplayDataset(cfg, native_nstep=True)


def _timed(rp, fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    t = np.zeros(8)
    rp.lib.a0_ckpt_last_timing(t.ctypes.data)
    return wall, t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=1_000_000)
    ap.add_argument("--out", default="profiles/reshard_b200.json")
    a = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    R = a.records
    cases = []
    with tempfile.TemporaryDirectory() as d:
        paths = []
        for seed in (1, 2):
            src = _shard(R)
            atari_fill(src, R, seed)
            paths.append(os.path.join(d, f"shard{seed}.a0ckpt"))
            src.save(paths[-1])
            del src
            torch.cuda.empty_cache()
        sizes = [os.path.getsize(p) for p in paths]
        plan = [("load", R, paths[:1]), ("merge_same", R, paths[:1]), ("merge_half", R // 2, paths[:1]),
                ("merge_double", 2 * R, paths[:1]), ("merge_two_into_double", 2 * R, paths)]
        for name, size, files in plan:
            dst = _shard(size)
            fn = (lambda: dst.load(files[0])) if name == "load" else (lambda: dst.load_merged(files))
            fn()                                                    # warm-up: first-use allocations
            wall, t = _timed(dst, fn)
            if name == "load":
                ph = dict(total_ms=t[0] / 1e3, validate_ms=t[1] / 1e3, file_read_ms=t[2] / 1e3, decode_restore_ms=t[3] / 1e3,
                          bytes_decoded=int(t[4]))
            else:
                ph = dict(total_ms=t[0] / 1e3, validate_ms=t[1] / 1e3, merge_plan_ms=t[2] / 1e3, decode_place_device_ms=t[3] / 1e3,
                          records_leaves_ms=t[4] / 1e3, file_read_hash_ms=t[7] / 1e3, bytes_decoded=int(t[5]),
                          bytes_placed=int(t[6]))
            line = dict(case=name, target_records=size, files=len(files), wall_ms=wall * 1e3, top=dst.top, **ph)
            print(json.dumps(line), flush=True)
            cases.append(line)
            del dst
            torch.cuda.empty_cache()
    out = dict(gpu=smi, records_per_file=R, checkpoint_bytes=sizes, frames="atari-like (tools/bench_checkpoint.py)",
               note="wall_ms: host clock around the call, ending in a device synchronise; second of two runs", cases=cases)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
