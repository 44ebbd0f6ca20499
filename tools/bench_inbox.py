"""The transition inbox (K9, agent0_b200/inbox.py) against what it replaces, on 84x84 frames (7056 B), E = 16 streams per
lane, a C51 shard of 1M records.

  commit_step        TransitionWriter.flush of one vector step (16 transitions, 16 new frames): host clock around the
                     H2D copy + K9a + synchronise; CUDA events around K9a alone
  commit_sample      the same for one sample()-sized slot (80 vector steps, 1280 transitions, ~1300 frames)
  drain_{1,4,8}      TransitionInbox.drain of one committed 1280-transition slot per lane: host clock around the whole
                     drain (K9b, its synchronise, validation, 80 append_steps calls per slot, K9c, then a synchronise);
                     CUDA events around K9b, and around the ingest + K9c (a span: host gaps between launches included)
  pickled_queue      the same 1280 transitions as per-step (streams, n_new, frames, action, reward, done) tuples pickled
                     by a spawned process into a multiprocessing queue; the learner's get + unpickle + 80 append_steps +
                     synchronise (the queue is filled ahead, so the producer's pickling is not on this clock)
  append_steps       in-process append_steps of the same 80 steps from host arrays + synchronise: the floor

K9a's bytes (metadata + frames, read from the device staging and written to the slot) over its event time is compared
with the copy bound 2 x bytes / 7.7 TB/s; the staging buffer of a sample-sized slot (9 MB) fits the 126 MB L2, so the
reads may be L2 hits.  One JSON object (card name, power limit and clocks read in the same run) to stdout and --out."""
import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from agent0_b200 import _lib  # noqa: E402
from agent0_b200.config import make_config  # noqa: E402
from agent0_b200.inbox import TransitionInbox, TransitionWriter  # noqa: E402
from agent0_b200.replay import ReplayDataset  # noqa: E402
from agent0_b200.ring_index import stack_delta  # noqa: E402
from agent0_b200.synth import SyntheticStreams  # noqa: E402

E, STEPS = 16, 80
HBM_BYTES_PER_S = 7.7e12


def _cfg(replay_size):
    cfg = make_config("c51", per=True, n_step=3, batch_size=32, double_q=True, dueling=True, num_envs=E,
                      replay_size=replay_size)
    cfg.actor.sample_steps = STEPS
    return cfg


def _steps(seed, n):
    env = SyntheticStreams(E, seed=seed, p_terminal=0.0, p_life_loss=0.0, p_truncated=0.0)   # one new frame per env
    obs, _ = env.reset()
    out = []
    for _ in range(n):
        a = env.sample_actions()
        nxt, r, term, trunc, info = env.step(a)
        out.append((obs, a, r, term, nxt))
        obs = nxt
    return out


def _as_native(steps):
    """Per step (streams, n_new, new frames, action, reward, done): what append_steps takes."""
    out = []
    for obs, a, r, d, nxt in steps:
        k = stack_delta(obs, nxt)
        new = np.concatenate([nxt[e, 4 - k[e]:] for e in range(E)])
        out.append((np.arange(E, dtype=np.int64), k, new, a, r, d))
    return out


def _stats(us):
    us = np.asarray(us, dtype=np.float64)
    return dict(mean_us=float(us.mean()), median_us=float(np.median(us)), p10_us=float(np.percentile(us, 10)),
                p90_us=float(np.percentile(us, 90)), n=int(us.size))


def _rearm(w, saved):
    w.packer.n_transitions, w.packer.n_steps, w.packer.n_frames = saved


def _commit(inbox, w, steps, iters):
    """Host and K9a times of committing ``steps`` (packed once, committed ``iters`` times; drained between)."""
    for s in steps:
        w.append_vector_step(*s)
    saved = (w.packer.n_transitions, w.packer.n_steps, w.packer.n_frames)
    nbytes = w.packer.nbytes()
    host, dev = [], []
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    st = _lib.stream_ptr(w.device)
    for i in range(iters):
        _rearm(w, saved)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        w.flush()
        host.append((time.perf_counter() - t0) * 1e6)
        inbox.drain()
        # K9a alone on the staging that flush left on the device
        _rearm(w, saved)
        ev0.record()
        _lib.check(w.lib.a0_tw_commit(w._h, w._dev.data_ptr(), *saved, w._status_mapped, st), "a0_tw_commit")
        ev1.record()
        torch.cuda.synchronize()
        assert int(w._status_host[0]) == _lib.TX_COMMITTED
        dev.append(ev0.elapsed_time(ev1) * 1e3)
        inbox.drain()
    _rearm(w, (0, 0, 0))
    moved = nbytes - 256
    k = _stats(dev)
    return dict(host=_stats(host), k9a=k, bytes=moved, k9a_bytes_per_s=moved / (k["median_us"] * 1e-6),
                copy_bound_us=2 * moved / HBM_BYTES_PER_S * 1e6,
                share_of_copy_bound=(2 * moved / HBM_BYTES_PER_S * 1e6) / k["median_us"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--replay", type=int, default=1_000_000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_inbox measures on the GPU"
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    res = dict(card=torch.cuda.get_device_name(0), nvidia_smi=smi, E=E, steps_per_slot=STEPS, frame_bytes=84 * 84)
    cfg = _cfg(args.replay)
    data = _steps(1, 2 * STEPS)
    slot_a, slot_b = data[:STEPS], data[STEPS:]

    rp = ReplayDataset(cfg, native_nstep=True)
    inbox = TransitionInbox(rp, 1, slots=2)
    w = TransitionWriter(inbox, lane=0)
    w.append_vector_step(*slot_a[0])
    w.flush()
    inbox.drain()
    res["commit_step"] = _commit(inbox, w, slot_b[:1], args.iters * 5)
    res["commit_sample"] = _commit(inbox, w, slot_b, args.iters)
    w.close()
    inbox.close()
    del rp

    for lanes in (1, 4, 8):
        res[f"drain_{lanes}"] = _drain(cfg, lanes, slot_a, slot_b, args.iters)

    native_a, native_b = _as_native(slot_a), _as_native(slot_b)
    res["append_steps"] = _append_floor(cfg, native_a, native_b, args.iters)
    res["pickled_queue"] = _pickled(cfg, native_a, native_b, args.iters)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


def _drain(cfg, lanes, slot_a, slot_b, iters):
    """Host clock around whole drains; CUDA events around K9b (a scan of the same committed slots, released unread)
    and around the ingest + K9c span."""
    rp = ReplayDataset(cfg, native_nstep=True)
    inbox = TransitionInbox(rp, lanes, slots=2)
    ws = [TransitionWriter(inbox, lane=l) for l in range(lanes)]
    for w in ws:
        for s in slot_a:
            w.append_vector_step(*s)
        w.flush()
    inbox.drain()
    for w in ws:
        for s in slot_b:
            w.append_vector_step(*s)
    saved = (ws[0].packer.n_transitions, ws[0].packer.n_steps, ws[0].packer.n_frames)
    st = _lib.stream_ptr(rp.device)
    e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    host, k9b, span = [], [], []

    def commit_all():
        for w in ws:
            _rearm(w, saved)
            w.flush()
        torch.cuda.synchronize()

    for i in range(iters + 2):
        commit_all()
        t0 = time.perf_counter()
        n = inbox.drain()
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        assert n == lanes * E * STEPS, n
        commit_all()
        e[0].record()
        _lib.check(inbox.lib.a0_tx_scan(inbox._h, inbox.slots, st), "a0_tx_scan")
        e[1].record()
        e[2].record()
        _lib.check(inbox.lib.a0_tx_release(inbox._h, st), "a0_tx_release")
        e[3].record()
        torch.cuda.synchronize()
        commit_all()
        ev_a, ev_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev_a.record()
        n = inbox.drain()
        ev_b.record()
        torch.cuda.synchronize()
        assert n == lanes * E * STEPS, n
        if i >= 2:
            host.append((t1 - t0) * 1e6)
            k9b.append(e[0].elapsed_time(e[1]) * 1e3)
            span.append(ev_a.elapsed_time(ev_b) * 1e3)
    return dict(transitions=lanes * E * STEPS, host_with_sync=_stats(host), k9b=_stats(k9b), device_span=_stats(span),
                k9c_us=e[2].elapsed_time(e[3]) * 1e3)


def _append_floor(cfg, native_a, native_b, iters):
    rp = ReplayDataset(cfg, native_nstep=True)
    rp.reset_streams(np.arange(E), np.zeros((E, 4, 84, 84), np.uint8))
    us = []
    for i in range(iters + 2):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for s in native_b:
            rp.append_steps(*s)
        torch.cuda.synchronize()
        if i >= 2:
            us.append((time.perf_counter() - t0) * 1e6)
    return dict(transitions=E * STEPS, host_with_sync=_stats(us))


def _producer(q, native, iters):
    for _ in range(iters):
        q.put(native)                              # pickled by the queue's feeder thread


def _pickled(cfg, native_a, native_b, iters):
    rp = ReplayDataset(cfg, native_nstep=True)
    rp.reset_streams(np.arange(E), np.zeros((E, 4, 84, 84), np.uint8))
    ctx = mp.get_context("spawn")
    q = ctx.Queue(maxsize=4)
    p = ctx.Process(target=_producer, args=(q, native_b, iters + 2), daemon=True)
    p.start()
    us = []
    try:
        for i in range(iters + 2):
            if i == 0:
                first = q.get(timeout=300)         # the child's start-up is not timed
                for s in first:
                    rp.append_steps(*s)
                torch.cuda.synchronize()
                continue
            time.sleep(0.05)                       # let the producer fill the queue ahead
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            msg = q.get(timeout=300)
            for s in msg:
                rp.append_steps(*s)
            torch.cuda.synchronize()
            if i >= 2:
                us.append((time.perf_counter() - t0) * 1e6)
        p.join(timeout=60)
    finally:
        if p.is_alive():
            p.terminate()
            p.join(timeout=10)
        if p.is_alive():
            p.kill()
            p.join(timeout=10)
    return dict(transitions=E * STEPS, bytes_pickled=int(sum(x.nbytes for s in native_b for x in s)),
                host_with_sync=_stats(us))


if __name__ == "__main__":
    main()
