"""Shard checkpoint phases on the device (a0_ckpt_save / a0_ckpt_load) against liblz4 on the host.

A C51 shard of --records records is filled with synth.fill_shard_synthetic (noise frames: every group is stored raw)
or, with --frames atari, with device-made "background + rectangles" frames that compress the way Atari frames do.
One JSON line per fill: the save and load phases of a0_ckpt_last_timing, K7's device time and bytes per frame, and
LZ4_compress_default of the system liblz4 over a sample of the same groups on one core and on every core.  The
checkpoint goes to a temporary directory; --out also writes the lines to a file."""
import argparse
import ctypes as C
import json
import multiprocessing as mp
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from agent0_b200 import _lib  # noqa: E402
from agent0_b200.config import make_config  # noqa: E402
from agent0_b200.replay import ReplayDataset  # noqa: E402
from agent0_b200.synth import fill_shard_synthetic  # noqa: E402
from oracle import cpu_path as CP  # noqa: E402


def atari_fill(rp, records, seed):
    """fill_shard_synthetic's stream structure with Atari-like frames made on the device."""
    g = torch.Generator(device=rp.device).manual_seed(seed)
    H, W = rp.frame_shape

    def frames(k):
        f = torch.randint(0, 64, (k, 1, 1), device=rp.device, generator=g, dtype=torch.int32).expand(k, H, W).clone()
        ys = torch.arange(H, device=rp.device).view(1, H, 1)
        xs = torch.arange(W, device=rp.device).view(1, 1, W)
        for _ in range(6):
            y0, x0 = (torch.randint(0, n, (k, 1, 1), device=rp.device, generator=g) for n in (H, W))
            h, w = (torch.randint(1, 16, (k, 1, 1), device=rp.device, generator=g) for _ in range(2))
            v = torch.randint(64, 256, (k, 1, 1), device=rp.device, generator=g, dtype=torch.int32)
            f = torch.where((ys >= y0) & (ys < y0 + h) & (xs >= x0) & (xs < x0 + w), v, f)
        return f.to(torch.uint8).view(k, -1)

    E = 16
    rng = np.random.RandomState(seed)
    rp.reset_streams(np.arange(E), frames(4 * E))
    T = max(1, min(rp.index.max_chunk // E, 4096))
    done = 0
    while done < records:
        m = T * E
        n_new = np.where(rng.rand(m) < 0.01, 4, 1).astype(np.int64)
        rp.append_steps(np.tile(np.arange(E, dtype=np.int64), T), n_new, frames(int(n_new.sum())), rng.randint(0, 4, m),
                        rng.choice([-1.0, 0.0, 1.0], m), rng.rand(m) < 0.005)
        done += m
    torch.cuda.synchronize(rp.device)


_GROUPS = []


def _compress_range(r):
    z = CP.lz4()
    return sum(len(z.compress(_GROUPS[i])) for i in range(*r))


def host_lz4(groups, procs):
    """Seconds and compressed bytes of LZ4_compress_default over ``groups`` in ``procs`` forked processes (the groups
    are inherited, not pickled; the pool is started before the clock)."""
    _GROUPS[:] = groups
    k = len(groups)
    ranges = [(k * i // procs, k * (i + 1) // procs) for i in range(procs)]
    if procs == 1:
        return _timed(lambda: _compress_range((0, k)))
    with mp.get_context("fork").Pool(procs) as pool:
        pool.map(_compress_range, [(0, 0)] * procs)
        return _timed(lambda: sum(pool.map(_compress_range, ranges)))


def _timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return time.perf_counter() - t0, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--records", type=int, default=1_000_000)
    ap.add_argument("--frames", default="noise,atari")
    ap.add_argument("--host-groups", type=int, default=4096)
    ap.add_argument("--out")
    a = ap.parse_args()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    lines = []
    for kind in a.frames.split(","):
        cfg = make_config("c51", per=True, n_step=3, batch_size=32, replay_size=a.records, double_q=True, dueling=True)
        src = ReplayDataset(cfg, native_nstep=True)
        if kind == "atari":
            atari_fill(src, a.records, 1)
        else:
            fill_shard_synthetic(src, a.records, 16, 1)
        lib, t = src.lib, np.zeros(8)
        with tempfile.TemporaryDirectory() as d:
            path = os.path.join(d, "shard.a0ckpt")
            src.save(path)                                  # warm-up: first-use allocations and attributes
            src.save(path)
            lib.a0_ckpt_last_timing(t.ctypes.data)
            save = dict(total_ms=t[0] / 1e3, encode_device_ms=t[1] / 1e3, compact_d2h_device_ms=t[2] / 1e3,
                        file_write_ms=t[3] / 1e3, wait_copy_ms=t[6] / 1e3, frame_bytes=int(t[4]), blob_bytes=int(t[5]))
            size = os.path.getsize(path)
            dst = ReplayDataset(cfg, native_nstep=True)
            subprocess.run(["sync"])
            t0 = time.perf_counter()
            dst.load(path)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            lib.a0_ckpt_last_timing(t.ctypes.data)
            load = dict(total_ms=t[0] / 1e3, validate_ms=t[1] / 1e3, file_read_ms=t[2] / 1e3, decode_restore_ms=t[3] / 1e3,
                        wall_ms=wall * 1e3)
            same = bool(torch.equal(src.tree, dst.tree)) and src.top == dst.top
            # liblz4 on the host over a sample of the same groups (the first --host-groups of the window)
            hfs = src.index.head_fs
            lo = max(0, hfs - src.index.NF)
            k = min(a.host_groups, (hfs - lo) // 8)
            pos = (torch.arange(lo, lo + 8 * k, device=src.device) % src.index.NF)
            host = src.frames[pos].view(k, -1).cpu().numpy()
            groups = [host[i].tobytes() for i in range(k)]
            cores = os.cpu_count()
            t1, c1 = host_lz4(groups, 1)
            tn, cn = host_lz4(groups, cores)
            gb = k * 8 * src.F / 1e9
            dev_gbs = save["frame_bytes"] / 1e9 / (save["encode_device_ms"] / 1e3)
        line = dict(frames=kind, records=a.records, gpu=smi, checkpoint_bytes=size, save=save, load=load, resumed_identical=same,
                    k7=dict(GB_per_s=dev_gbs, bytes_per_frame=save["blob_bytes"] / max(1, save["frame_bytes"] / src.F)),
                    liblz4_host=dict(sample_groups=k, cores=cores, one_core_GB_per_s=gb / t1, all_cores_GB_per_s=gb / tn,
                                     bytes_per_frame=cn / (8 * k)))
        print(json.dumps(line), flush=True)
        lines.append(line)
        del src, dst
        torch.cuda.empty_cache()
    if a.out:
        with open(a.out, "w") as f:
            for ln in lines:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
