#!/usr/bin/env python
"""bench.py -- replay sample+target throughput of the agent0 deepq hot path on B200.

  python bench.py --gpus N --steps K --warmup W            our CUDA path (one rank per GPU)
  python bench.py --impl reference --steps K --warmup W    the reference's own CPU pipeline (oracle/_ref: the unmodified
                                                           reference; the restated port where it cannot run)

One "step" = the inner loop of the reference's Trainer.step (agent0/deepq/trainer.py:82-104) with
the CNN excluded (network outputs pre-generated): draw L = learner_steps batches of B transitions
from the prioritized shard (K2a, one launch), gather them (K3, one launch: stack reconstruction +
n-step return), run the fused target/loss kernel once per batch (K4, L launches) and write the new
priorities (K2b, one launch).  Headline workload = BASELINE.json configs[1]: C51 51 atoms, PER,
n_step=3, double+dueling, batch 32, L=20, 1 M-transition ring of synthetic 84x84 uint8 frames.
`value` times that loop as a CUDA graph with everything resident in HBM; `e2e` times the same work
through the public Python API with new transitions arriving from pinned host memory every step
(replay ratio 8 samples per insert, agent0/deepq/config.py) and the losses read back to the host.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

F_BYTES = 84 * 84
METRIC = "replay_sample_target_transitions_per_sec"
UNIT = "transitions/s"

# BASELINE.json configs, as (algo, per, n_step, double, B, extra)
WORKLOADS = {
    "c51_b32": dict(algo="c51", per=True, n=3, double=True, B=32, desc="configs[1]: C51 51 atoms, PER, n_step=3, double+dueling, batch 32"),
    "dqn_b32_uniform": dict(algo="dqn", per=False, n=1, double=False, B=32, desc="configs[0]: DQN, uniform replay, n_step=1, batch 32"),
    "qr_b512": dict(algo="qr", per=True, n=3, double=True, B=512, desc="configs[2]: QR-DQN 200 quantiles, PER, batch 512"),
    "iqn_b512": dict(algo="iqn", per=True, n=3, double=True, B=512, desc="configs[2]: IQN 64x64 taus, PER, batch 512"),
    "fqf_b512": dict(algo="fqf", per=True, n=3, double=True, B=512, desc="configs[3]: FQF 32 fractions, PER, batch 512"),
    "mdqn_b512": dict(algo="mdqn", per=True, n=3, double=False, B=512, desc="configs[3]: M-DQN, PER, batch 512"),
    "c51_b512": dict(algo="c51", per=True, n=3, double=True, B=512, desc="C51, PER, n_step=3, batch 512"),
}


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=200)
    p.add_argument("--warmup", type=int, default=10)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--workload", default="c51_b32", choices=sorted(WORKLOADS))
    p.add_argument("--ring", type=int, default=1_000_000, help="transitions per GPU shard")
    p.add_argument("--total-ring", type=int, default=0, help="if set, shard this many transitions over the GPUs (configs[4]: 8M)")
    p.add_argument("--learner-steps", type=int, default=20)
    p.add_argument("--actions", type=int, default=4)
    p.add_argument("--no-extra", action="store_true", help="skip the secondary workloads and sweeps")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-learner", action="store_true", help="skip the data-parallel learner-step measurement (learner_scaling)")
    p.add_argument("--no-graph", action="store_true")
    p.add_argument("--torch-rng", action="store_true", help="uniforms from torch.Tensor.uniform_ (one more launch per step) instead of the sampler's own Philox")
    p.add_argument("--variant", type=int, default=0, help="K3 variant: 0 TMA ring, 1 LDG/STG, 2 TMA full staging, 3 TMA two CTAs per transition")
    p.add_argument("--cpu-entries", type=int, default=1_000_000, help="entries in the CPU arm's lz4 deque (replay.py:18: 1 M)")
    p.add_argument("--cpu-distinct", type=int, default=16384, help="distinct lz4 blobs behind those entries (the deque holds references)")
    p.add_argument("--min-seconds", type=float, default=0.25, help="secondary measurements (not value, not e2e.value): repeat their "
                   "blocks until this much time")
    p.add_argument("--dump-outputs", metavar="DIR", default=None, help="after the timed steps, write what the last timed step computed "
                   "(indices, IS weights, losses, gradients, the gathered batch) as DIR/<name>.npy (--impl ours)")
    p.add_argument("--gather-waves", default="auto", help="gather schedule of the step: auto (waves on a side stream, K4 of batch k waits "
                   "for its wave only), none (one gather launch before the first K4), or wave sizes in batches, e.g. 1,1,2,4,12")
    p.add_argument("--gather-window", default="auto", help="ordered fetch inside the gather waves: draws in flight beyond the completed ones (auto | 0 = no limit | n)")
    p.add_argument("--eager-waves", action="store_true", help="with --no-graph: issue the gather waves eagerly too (the ncu launch list of the "
                   "captured schedule; by default an eagerly issued step uses the single gather launch, see hotloop.ReplayTargetLoop)")
    p.add_argument("--no-k4-priority", action="store_true", help="K4 + K2b on the caller's stream instead of the loop's high-priority stream")
    p.add_argument("--no-pdl-at-joins", action="store_true", help="the K4 that joins a gather wave is launched without its programmatic-launch attribute")
    p.add_argument("--cpu-workers", type=int, default=-1, help="--impl reference DataLoader workers (-1: all cores)")
    a = p.parse_args()
    if a.steps < 1 or a.warmup < 0:
        p.error("--steps must be >= 1 and --warmup >= 0")
    if a.dump_outputs and a.impl != "ours":
        p.error("--dump-outputs writes what the CUDA path computed: --impl ours only")
    return a


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled every 200 ms during the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *a):
        if self.proc is not None:
            time.sleep(0.25)
            self.proc.terminate()
            self.thread.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------ our arm
def fill_shard(rp, transitions, E, seed, torch):
    from agent0_b200.synth import fill_shard_synthetic
    return fill_shard_synthetic(rp, transitions, E, seed)


def net_outputs(algo, total, A, torch, dev, seed=99):
    """Pre-generated network outputs (the CNN is excluded on both arms): N(0,1)*3 logits."""
    g = torch.Generator(device=dev).manual_seed(seed)
    rn = lambda *s: torch.randn(*s, device=dev, generator=g) * 3.0
    o = {"qsel": rn(total, A)}
    if algo in ("dqn", "mdqn"):
        o.update(online=rn(total, A), tgt_next=rn(total, A), tgt_cur=rn(total, A))
    elif algo == "c51":
        o.update(online=rn(total, A, 51), tgt_next=rn(total, A, 51), atoms=torch.linspace(-10, 10, 51, device=dev))
    elif algo == "qr":
        o.update(online=rn(total, A, 200), tgt_next=rn(total, A, 200))
    elif algo == "iqn":
        o.update(online=rn(total, 64, A), tgt_next=rn(total, 64, A), taus=torch.rand(total, 64, device=dev, generator=g))
    elif algo == "fqf":
        p = torch.softmax(torch.randn(total, 32, device=dev, generator=g), -1)
        taus = torch.cat((torch.zeros(total, 1, device=dev), torch.cumsum(p, -1)), -1)
        o.update(online=rn(total, 32, A), tgt_next=rn(total, 32, A), q_bar=rn(total, 31, A), taus=taus.contiguous(),
                 taus_hat=((taus[:, :-1] + taus[:, 1:]) / 2).contiguous())
    return o


def bytes_per_transition(n):
    """SURVEY 8d: K3 reads (S+n) distinct frames and writes 2S frames per transition."""
    return (4 + min(n, 4) + 8) * F_BYTES


def make_hotpath(rp, wl, L, A, torch, variant=0, waves=None):
    from agent0_b200.hotloop import ReplayTargetLoop
    waves = GATHER_WAVES if waves is None else (None if waves == "none" else waves)

    class HotPath(ReplayTargetLoop):
        """agent0_b200.hotloop.ReplayTargetLoop (the package's pre-bound form of the Trainer.step inner
        loop) plus what only the benchmark needs: synthetic network outputs, and pools of pre-drawn
        index sets and rotating output buffers so that back-to-back timed gathers neither re-read
        frames nor have their stores absorbed by L2."""

        def __init__(self):
            T = L * wl["B"]
            # timed gathers rotate over enough output buffers (>= ~1 GB) that stores are not absorbed by L2
            self.n_out = min(INNER, max(1, int(1e9 // (T * 8 * F_BYTES))))
            self.frames_pool = torch.empty(self.n_out, T, 8 * F_BYTES, dtype=torch.uint8, device=rp.device)
            super().__init__(rp, wl["algo"], wl["B"], L, A, net_outputs(wl["algo"], T, A, torch, rp.device), n_step=wl["n"],
                             double_q=wl["double"], per=wl["per"], variant=variant, discount=0.99, frames=self.frames_pool[0],
                             rng_seed=RNG_SEED, gather_waves=waves, pdl_at_joins=PDL_AT_JOINS,
                             gather_window=GATHER_WINDOW, k4_priority=K4_PRIORITY, waves_when_eager=EAGER_WAVES)
            self.wl, self.idx_pool = wl, None

        def draw_pool(self):
            """INNER independent index sets, so that back-to-back timed gathers never re-read frames."""
            self.idx_pool = torch.empty(INNER, self.total, dtype=torch.int64, device=self.dev)
            for i in range(INNER):
                self.u.uniform_(); self.sample()
                self.idx_pool[i].copy_(self.idx)

        def gather(self, count=None, variant=None, pool=None):
            if pool is None:
                return super().gather(count=count, variant=variant)
            return super().gather(self.idx_pool[pool % INNER].data_ptr(), self.frames_pool[pool % self.n_out].data_ptr(),
                                  count, variant)

        loss_k = ReplayTargetLoop.target_loss

        def step_fused_k4(self):
            self.step(fused_k4=True)

    return HotPath()


def HotPath(rp, wl, L, A, torch, variant=0, waves=None):
    return make_hotpath(rp, wl, L, A, torch, variant, waves)


def time_graphed(hp, steps, warmup, torch, use_graph, barrier, step_fn=None, min_seconds=0.0, reduce_max=None, stats=None):
    """Device time of ONE block of exactly ``steps`` steps (CUDA events on the launching stream, barrier +
    synchronize on both sides), after SETTLE + ``warmup`` untimed steps.  With ``min_seconds`` > 0 (the secondary
    measurements) the block is repeated until that much device time has been measured and the MEDIAN block is
    returned; the headline ``value`` times one block, so that --steps is the number of timed steps and the state
    after them (--dump-outputs) is fixed by the arguments.  ``stats`` receives every block's seconds.  ``reduce_max(t)``: max over ranks of one block's time
    (so every rank sees the same totals and runs the same number of blocks)."""
    step_fn = step_fn or hp.step
    hp.rp.push_dynamic()
    for _ in range(3):
        step_fn()
    torch.cuda.synchronize()
    runner = step_fn
    if use_graph:
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            step_fn()
        runner = g.replay
    for _ in range(SETTLE + warmup):
        runner()
    torch.cuda.synchronize()
    blocks, total = [], 0.0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    while True:
        barrier()
        e0.record()
        for _ in range(steps):
            runner()
        e1.record()
        torch.cuda.synchronize()
        barrier()
        dt = e0.elapsed_time(e1) / 1e3
        if reduce_max is not None:
            dt = reduce_max(dt)
        blocks.append(dt)
        total += dt
        if total >= min_seconds or len(blocks) >= 2000:
            break
    if stats is not None:
        stats.extend(blocks)
    return float(np.median(blocks))


def _sample_rows(total, row_bytes, budget, seed):
    """All rows, or a fixed seeded sample of them that fits ``budget`` bytes."""
    n = max(1, min(total, budget // row_bytes))
    return np.arange(total) if n == total else np.sort(np.random.default_rng(seed).choice(total, n, replace=False))


def dump_outputs(hp, out_dir, torch):
    """--dump-outputs: what the last step of ``hp`` computed, as out_dir/<name>.npy in float32 / float64 (integers as
    float64, exact): the drawn indices and IS weights, per-sample losses, gradients w.r.t. the online output, the
    gathered batch and the priorities K2b wrote.  Under 64 MB in all: the gradients are cut to a seeded row sample above
    32 MB, the gathered frame stacks (8 x 84 x 84 u8 per transition) to a seeded sample of 16 MB (*_rows.npy: which)."""
    torch.cuda.synchronize()
    T = hp.total
    f64 = lambda t: t.cpu().numpy().astype(np.float64)
    f32 = lambda t: t.cpu().numpy().astype(np.float32)
    out = {"indices": f64(hp.idx), "weights": f32(hp.w), "loss": f32(hp.loss), "actions": f64(hp.act),
           "returns": f64(hp.r64), "terminals": f32(hp.d32), "bootstrap": f64(hp.boot),
           "priorities": f32(hp.rp.priority.leaves()[hp.idx]), "max_priority": f32(hp.rp.max_p_tensor)}
    grad = hp.grad.view(T, -1)
    g_rows = _sample_rows(T, grad.shape[1] * 4, 32 << 20, 1)
    out["grad"] = f32(grad[torch.from_numpy(g_rows).to(grad.device)].view(-1, *hp.grad.shape[1:]))
    if len(g_rows) < T:
        out["grad_rows"] = g_rows.astype(np.float64)
    if hp.frac is not None:                                   # FQF: fraction-loss outputs
        out["fraction_loss"], out["fraction_grad"] = f32(hp.frac), f32(hp.gtau)
    fr_rows = _sample_rows(T, hp.frames.shape[1] * 4, 16 << 20, 2)
    out["frames"] = f32(hp.frames[torch.from_numpy(fr_rows).to(hp.frames.device)])
    out["frames_rows"] = fr_rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def block_stats(blocks, units_per_block):
    """median / p10 / p90 of the per-block rates (p10 / p90 only when there is more than one block)."""
    r = np.sort(units_per_block / np.asarray(blocks, dtype=np.float64))
    q = lambda p: float(r[min(len(r) - 1, int(round(p * (len(r) - 1))))])
    out = {"blocks": len(r), "timed_region_s": round(float(np.sum(blocks)), 4), "rate_median": round(float(np.median(r)), 1)}
    if len(r) > 1:
        out.update(rate_p10=round(q(0.1), 1), rate_p90=round(q(0.9), 1))
    return out


EMIT = print
INNER = 20
SETTLE = 200             # untimed steps before the --warmup ones: the first ~150 replays of a freshly captured step run 1-2 %
                         # slower (profiles/settle_first_replays.txt); a fixed count keeps the state deterministic
GATHER_WAVES = "auto"    # --gather-waves
PDL_AT_JOINS = True      # --no-pdl-at-joins
GATHER_WINDOW = "auto"   # --gather-window
K4_PRIORITY = True       # --no-k4-priority
EAGER_WAVES = False      # --eager-waves
RNG_SEED = 20261017      # the sampler draws its own uniforms (Philox inside K2a); None: torch's uniform_ + a0_pt_sample


def capture_step(hp, torch):
    hp.rp.push_dynamic()
    for _ in range(3):
        hp.step()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        hp.step()
    return g


def time_kernel(fn, reps, torch):
    """Average device duration of one launch: INNER back-to-back launches ``fn(i)`` (i selects
    distinct pre-drawn inputs where that matters) captured into one CUDA graph so the host launch
    path is not on the clock; CUDA events on the launching stream around the replays."""
    fn(0)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for i in range(INNER):
            fn(i)
    g.replay()
    torch.cuda.synchronize()
    rounds = max(1, reps // INNER)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(rounds):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3 / (rounds * INNER)


def e2e_cabi(hp, steps, warmup, torch, graph=True, depth=2, copy_stream=True, fused=True, min_seconds=0.0, stats=None):
    """The headline end-to-end number: one Trainer.step-shaped pass driven through the C ABI with
    HOST buffers.  Per step: new transitions (replay ratio 8 samples per insert) are ingested from
    page-locked host memory (a0_rb_ingest_steps_dyn: index update, H2D DMA, K2b marks + K1 in one
    launch, which also publishes the shard's top/beta to the device); the L batches are drawn,
    gathered, run through K4 and written back to the tree by replaying ONE CUDA graph of the
    C-ABI launches (``graph=False``: the same launches issued eagerly); the per-sample losses and
    indices reach page-locked host memory -- stored there by the K2b launch that reads them
    (a0_pt_update_report) -- and are read by the host.

    ``fused=False`` is the same loop with the separate pieces: a0_rb_ingest_steps, an
    a0_rb_set_dynamic launch, and two device-to-host copies queued behind the graph.

    depth=1: the host waits for the step's losses before it starts the next step.  depth=2: the
    result buffers are double-buffered -- the host reads step s-1's losses while the device runs
    step s (the reference's own pump is asynchronous too: 2 worker processes and a 3-deep
    prefetch queue, utils.py:59-61).  Every step's H2D input copy and D2H result read, and the
    final drain, are inside the timed region either way.  ``copy_stream``: the ingest's H2D DMA
    runs on the shard's copy stream so it overlaps the previous step's kernels.
    Wall clock around a block of ``steps`` steps; the block is repeated until ``min_seconds`` of wall clock
    have been measured and the median block rate is returned (``stats`` receives every block's seconds)."""
    rp, L, B = hp.rp, hp.L, hp.B
    total = hp.total
    new_per_step = max(16, total // 8)
    E = 16
    rng = np.random.RandomState(3)
    host_frames = [torch.randint(0, 256, (new_per_step, F_BYTES), dtype=torch.uint8).pin_memory() for _ in range(depth + 1)]
    streams = np.arange(new_per_step, dtype=np.int64) % E
    ones_new = np.ones(new_per_step, dtype=np.int64)
    actions = rng.randint(0, 4, new_per_step).astype(np.int64)
    zr, zd = np.zeros(new_per_step), np.zeros(new_per_step, dtype=bool)
    if fused:
        rep = hp.bind_report(depth)
        idx_host, loss_host = [r[0] for r in rep], [r[1] for r in rep]
    else:
        loss_host = [torch.empty(total, dtype=torch.float32).pin_memory() for _ in range(depth)]
        idx_host = [torch.empty(total, dtype=torch.int64).pin_memory() for _ in range(depth)]
    done_ev = [torch.cuda.Event() for _ in range(depth)]
    h2d = new_per_step * (F_BYTES + 14 * 4 + 4 + 4)
    d2h = total * (4 + 8)

    g = None
    if graph and fused:
        hp.capture_reporting()
    elif graph:
        g = capture_step(hp, torch)
    else:
        hp.graphs, hp.graph = [], None
    acc = [0.0, 0]

    def consume(slot):
        done_ev[slot].synchronize()
        acc[0] += float(loss_host[slot][0]) + float(loss_host[slot][-1])     # the host reads the result
        acc[1] = max(acc[1], int(idx_host[slot][0]))

    def run(n):
        for s in range(n):
            slot = s % depth
            if s >= depth:
                consume(slot)                       # step s-depth: its buffers are reused below
            rp.append_steps(streams, ones_new, host_frames[s % (depth + 1)], actions, zr, zd, pinned_stable=True,
                            copy_stream=copy_stream, publish_dynamic=fused)
            if fused:
                hp.run(slot=slot, publish=False)
            else:
                rp.push_dynamic()
                if g is not None:
                    g.replay()
                else:
                    hp.step()
                loss_host[slot].copy_(hp.loss, non_blocking=True)
                idx_host[slot].copy_(hp.idx, non_blocking=True)
            done_ev[slot].record()
        for s in range(max(0, n - depth), n):
            consume(s % depth)

    run(warmup)
    torch.cuda.synchronize()
    blocks, spent = [], 0.0
    while True:
        t0 = time.perf_counter()
        run(steps)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        blocks.append(dt)
        spent += dt
        if spent >= min_seconds or len(blocks) >= 2000:
            break
    assert all(torch.isfinite(x).all() for x in loss_host) and acc[1] < rp.size and np.isfinite(acc[0])
    if fused:       # what reached the host is what the device holds
        last = (steps - 1) % depth
        assert torch.equal(loss_host[last], hp.loss.cpu()) and torch.equal(idx_host[last], hp.idx.cpu())
    if stats is not None:
        stats.extend(blocks)
    return total * steps / float(np.median(blocks)), h2d, d2h


def reference_entries(count, n_step, E=16, seed=77):
    """``count`` reference actor tuples (lz4.block.compress(concat(st, st_next)), a, r, d) (agent.py:78-81) from the
    synthetic Atari-like stream, in the actor's order (step-major, env-minor)."""
    from agent0_b200.synth import record_stream
    from oracle import cpu_path as CP, reference_replay as OR_
    s_ = record_stream(E, count // E + n_step + 2, seed=seed)
    fr_, a_, r_, d_ = OR_.pack_nstep(s_["obs"], s_["action"], s_["reward"], s_["done"], n_step, 0.99)
    z = CP.lz4()
    return [(z.compress(fr_[i].tobytes()), a_[i], r_[i], d_[i]) for i in range(count)]


def e2e_extend(wl, L, A, steps, torch, min_seconds, entries, per_step=1280, ring=200_000):
    """The drop-in shape of a Trainer.step (trainer.py:74-104), end to end through the public API with HOST
    inputs: ``replay.extend(list of the actor's lz4 tuples)`` -- 80 steps x 16 envs = 1280 entries, what the
    reference actor ships per step (config.py:111-112) -- then the L batches drawn, gathered, run through K4 and
    written back (one CUDA-graph replay), losses + indices read by the host (double-buffered).  The compressed
    bytes cross PCIe, K6 decodes and de-duplicates on the device.  Returns sampled transitions per second,
    inserted transitions per second, and the extend() call's own milliseconds."""
    from agent0_b200.config import make_config
    from agent0_b200.replay import ReplayDataset
    cfg = make_config(wl["algo"], per=wl["per"], n_step=wl["n"], batch_size=wl["B"], replay_size=ring, double_q=wl["double"],
                      dueling=True, num_envs=16, action_dim=A)
    rq = ReplayDataset(cfg)                                   # reference entries: already n-step folded
    calls = len(entries) // per_step
    assert calls >= 4
    rq.extend(entries[:per_step])
    from agent0_b200.hotloop import ReplayTargetLoop
    hp = ReplayTargetLoop(rq, wl["algo"], wl["B"], L, A, net_outputs(wl["algo"], L * wl["B"], A, torch, rq.device), n_step=1,
                          double_q=wl["double"], per=wl["per"], discount=0.99, rng_seed=RNG_SEED)
    rep = hp.bind_report(2)
    hp.capture_reporting()
    ev = [torch.cuda.Event() for _ in range(2)]
    acc = [0.0]
    ext_ms = []

    def run(n, c0):
        for s in range(n):
            slot = s % 2
            if s >= 2:
                ev[slot].synchronize()
                acc[0] += float(rep[slot][1][0])
            c = (c0 + s) % calls
            t0 = time.perf_counter()
            rq.extend(entries[c * per_step:(c + 1) * per_step])
            ext_ms.append((time.perf_counter() - t0) * 1e3)
            hp.run(slot=slot)
            ev[slot].record()
        for s in range(max(0, n - 2), n):
            ev[s % 2].synchronize()
            acc[0] += float(rep[s % 2][1][0])

    run(3, 1)
    torch.cuda.synchronize()
    ext_ms.clear()
    blocks, spent, c0 = [], 0.0, 4
    while True:
        t0 = time.perf_counter()
        run(steps, c0)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        blocks.append(dt); spent += dt; c0 += steps
        if spent >= min_seconds or len(blocks) >= 200:
            break
    assert np.isfinite(acc[0])
    med = float(np.median(blocks))
    return {"value": round(hp.total * steps / med, 1), "inserts_per_s": round(per_step * steps / med, 1),
            "extend_ms": round(float(np.median(ext_ms)), 3), "entries_per_extend": per_step,
            "h2d_bytes_per_step": int(sum(len(e[0]) for e in entries[:per_step]) + per_step * 24),
            "d2h_bytes_per_step": hp.total * 12 + per_step * 12, "timing": rq.extend_timing(), "blocks": len(blocks)}




def e2e_loop(rp, wl, L, A, steps, warmup, torch):
    """Same work through the public API with host buffers: append new transitions from pinned host
    memory (K1), sample+gather, K4 per batch, update priorities, read losses+indices back."""
    from agent0_b200 import losses as LS
    dev, B, algo = rp.device, wl["B"], wl["algo"]
    total = L * B
    o = net_outputs(algo, total, A, torch, dev)
    new_per_step = max(16, total // 8)            # replay ratio: 8 samples per inserted transition
    E = 16
    rng = np.random.RandomState(3)
    host_frames = torch.randint(0, 256, (new_per_step, F_BYTES), dtype=torch.uint8).pin_memory()
    streams = np.arange(new_per_step, dtype=np.int64) % E
    gam = float(np.float32(0.99 ** wl["n"]))
    h2d = new_per_step * (F_BYTES + 14 * 4 + 4)
    d2h = total * (4 + 8)

    from agent0_b200.replay import split_batches
    os_ = {k: (v.split(B) if v.dim() and v.shape[0] == total else v) for k, v in o.items()}
    use_qsel = wl["double"] or algo in ("iqn", "fqf")
    kw = dict(max_p=rp.max_p_tensor)
    ones_new = np.ones(new_per_step, dtype=np.int64)
    zr, zd = np.zeros(new_per_step), np.zeros(new_per_step, dtype=bool)

    def one():
        # the step's inputs come from pinned host memory; the ingest DMA reads the caller's buffer directly
        rp.append_steps(streams, ones_new, host_frames, rng.randint(0, 4, new_per_step), zr, zd, pinned_stable=True)
        b = rp.sample(B, k_batches=L)
        outs = []
        for k, bk in enumerate(split_batches(b, B)):
            cm = (bk.actions, bk.rewards_f32, bk.terminals_f32, bk.weights, gam)
            qs = os_["qsel"][k] if use_qsel else None
            if algo == "dqn":
                r = LS.dqn_loss(os_["online"][k], os_["tgt_next"][k], *cm, qsel=qs, **kw)
            elif algo == "mdqn":
                r = LS.mdqn_loss(os_["online"][k], os_["tgt_next"][k], os_["tgt_cur"][k], *cm, **kw)
            elif algo == "c51":
                r = LS.c51_loss(os_["online"][k], os_["tgt_next"][k], os_["atoms"], *cm, -10.0, 10.0, qsel=qs, **kw)
            elif algo == "qr":
                r = LS.qr_loss(os_["online"][k], os_["tgt_next"][k], *cm, qsel=qs, **kw)
            elif algo == "iqn":
                r = LS.iqn_loss(os_["online"][k], os_["taus"][k], os_["tgt_next"][k], qs, *cm, **kw)
            else:
                r = LS.fqf_loss(os_["online"][k], os_["taus"][k], os_["taus_hat"][k], os_["tgt_next"][k], os_["q_bar"][k], qs,
                                *cm, **kw)
            outs.append(r.loss)
        loss = torch.cat(outs)
        rp.update_priority(b.indices, loss)
        return loss.cpu(), b.indices.cpu()       # what BaseLearner.train returns (agent.py:163-169)

    for _ in range(warmup):
        one()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return total * steps / dt, h2d, d2h


def shared_config(wl, L, A, ring, args):
    """The keys BOTH arms print under ``config`` (same workload, same sizes): the driver compares them."""
    return {"workload": wl["desc"], "learner_steps_per_step": L, "transitions_per_step_per_gpu": L * wl["B"],
            "ring_transitions_per_gpu": ring, "actions": A, "cpu_entries": args.cpu_entries,
            "l2": "inputs larger than L2 (random reads over the multi-GB frame ring; K3's timed launches rotate over > 700 MB "
                  "of outputs and 20 index sets); not applicable to the CPU arm"}


def make_shard(wl, ring, A, rank, torch, variant=0):
    from agent0_b200.config import make_config
    from agent0_b200.replay import ReplayDataset
    cfg = make_config(wl["algo"], per=wl["per"], n_step=wl["n"], batch_size=wl["B"], replay_size=ring,
                      double_q=wl["double"], dueling=True, num_envs=16, action_dim=A)
    t0 = time.perf_counter()
    rp = ReplayDataset(cfg, native_nstep=True, gather_variant=variant)
    fill_shard(rp, ring, 16, 1234 + rank, torch)
    return rp, time.perf_counter() - t0


def run_ours(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py (ours) needs a GPU: there is no CPU fallback"
    torch.cuda.set_device(local)
    if world > 1:
        from agent0_b200.dist import init_nccl
        init_nccl(local, high_priority=os.environ.get("A0_NCCL_HIGH_PRIORITY", "1") != "0")
    barrier = (lambda: dist.barrier()) if world > 1 else (lambda: None)

    def reduce_max(x):
        if world == 1:
            return x
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    wl = WORKLOADS[args.workload]
    L, A = args.learner_steps, args.actions
    global RNG_SEED, GATHER_WAVES, PDL_AT_JOINS, GATHER_WINDOW, K4_PRIORITY, EAGER_WAVES
    EAGER_WAVES = bool(args.eager_waves)
    GATHER_WINDOW = "auto" if args.gather_window == "auto" else int(args.gather_window)
    K4_PRIORITY = not args.no_k4_priority
    PDL_AT_JOINS = not args.no_pdl_at_joins
    GATHER_WAVES = None if args.gather_waves == "none" else ("auto" if args.gather_waves == "auto" else [int(x) for x in args.gather_waves.split(",")])
    if args.torch_rng:
        RNG_SEED = None
    elif RNG_SEED is not None:
        RNG_SEED += rank
    ring = args.total_ring // world if args.total_ring else args.ring
    rp, t_fill = make_shard(wl, ring, A, rank, torch, args.variant)
    hp = HotPath(rp, wl, L, A, torch, variant=args.variant)

    blocks = []
    with ClockSampler(local) as clk:     # exactly --steps timed steps: one block
        secs = time_graphed(hp, args.steps, args.warmup, torch, not args.no_graph, barrier, reduce_max=reduce_max, stats=blocks)
    if args.dump_outputs and rank == 0:
        dump_outputs(hp, args.dump_outputs, torch)
    total = hp.total
    value = total * args.steps * world / secs
    timing = block_stats(blocks, total * args.steps * world)
    launches_per_step = hp.launches_per_step
    wave_sizes = [w[1] for w in hp.waves] if hp.waves else None
    wave_window = hp.window if hp.waves else None

    # ---- roofline of the dominant kernel (K3), same launch shape, fresh indices every launch -------
    hp.draw_pool()
    k3 = time_kernel(lambda i: hp.gather(pool=i), max(200, min(args.steps, 400)), torch)
    bpt = bytes_per_transition(wl["n"])
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = bpt * total / k3 / 1e9
    traffic, traffic_src = None, None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "k3_traffic.json")))
        traffic, traffic_src = tj.get(f"{total}"), tj.get("source")
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": ["a0_k3_gather_tma", "a0_k3_gather_ldg", "a0_k3_gather_tma_full", "a0_k3_gather_tma_split"][args.variant],
                "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback",
                "bytes_per_launch": bpt * total, "launch_us": round(k3 * 1e6, 2), "transitions_per_launch": total}

    # ---- e2e through the public API -----------------------------------------------------------------
    barrier()
    e2e_blocks = []
    e2e_v, h2d, d2h = e2e_cabi(hp, args.steps, SETTLE + 5, torch, graph=not args.no_graph, depth=2, copy_stream=True,
                               stats=e2e_blocks)   # its graphs are freshly captured too
    e2e_timing = block_stats(e2e_blocks, total * args.steps)
    side = [0.0, 0.0, 0.0, 0.0]
    if not args.no_extra:
        short = min(args.min_seconds, 0.1)
        barrier()
        side[0], _, _ = e2e_cabi(hp, args.steps, 5, torch, graph=not args.no_graph, depth=1, copy_stream=False, min_seconds=short)
        barrier()
        side[1], _, _ = e2e_cabi(hp, args.steps, 5, torch, graph=False, depth=2, copy_stream=True, min_seconds=short)
        barrier()
        side[2], _, _ = e2e_cabi(hp, args.steps, 5, torch, graph=not args.no_graph, depth=2, copy_stream=True, fused=False, min_seconds=short)
        barrier()
        side[3], _, _ = e2e_loop(rp, wl, L, A, max(10, args.steps), 3, torch)
    t = torch.tensor([e2e_v] + side, device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    e2e_v, e2e_sync, e2e_eager, e2e_sep, e2e_py = (float(x) for x in t.tolist())

    extra, configs, ext = {}, [], None
    if world > 1:
        extra["grad_allreduce"] = grad_allreduce_probe(torch, dist, world, barrier, L)
        extra["weight_broadcast"] = weight_broadcast_probe(torch, dist, world, barrier, A)
    if not args.no_extra and rank == 0 and world == 1:
        entries = reference_entries(5 * 1280, wl["n"])
        ext = e2e_extend(wl, L, A, max(4, min(args.steps, 20)), torch, args.min_seconds, entries)
        configs.append({"workload": args.workload, "desc": wl["desc"], "value": round(value, 1),
                        "ms_per_step": round(secs / args.steps * 1e3, 5), "k3_frac": roofline["frac"], "ring": ring})
        extra = extras(rp, args, torch, peak, configs, entries)
        del rp, hp
        torch.cuda.empty_cache()
        extras_other_shards(args, torch, peak, configs)
    learner = None
    if not args.no_extra and not args.no_learner:
        try:
            learner = learner_scaling(args, torch, dist, world, rank, barrier, reduce_max, A)
        except Exception as e:      # measurement only: the replay+target line must still be printed
            learner = {"error": repr(e)[:400]}
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline(wl, L, A, args, workers=0)

    if rank == 0:
        e2e = {"value": round(e2e_v, 1), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "timing": e2e_timing,
               "path": "agent0_b200 public API over the C ABI (ReplayDataset.append_steps + hotloop.ReplayTargetLoop): ingest from pinned host buffers "
                       "(H2D DMA on the shard's copy stream; marks + append + top/beta publication in one launch) + one CUDA-graph "
                       "replay of the C-ABI launches per step; losses and indices stored by the K2b launch into double-buffered "
                       "mapped pinned host memory (a0_pt_update_report), the host reads step s-1's result while step s runs "
                       "(final drain inside the timed region)"}
        if not args.no_extra:
            e2e.update({"separate_launches_value": round(e2e_sep, 1),
                        "separate_launches_path": "same loop with a0_rb_set_dynamic as its own launch and two device-to-host copies queued behind the graph",
                        "sync_every_step_value": round(e2e_sync, 1),
                        "sync_every_step_path": "same, but the host waits for each step's losses before starting the next (depth 1)",
                        "cabi_eager_value": round(e2e_eager, 1),
                        "python_api_value": round(e2e_py, 1),
                        "python_api_path": "ReplayDataset.append_steps/sample/update_priority + agent0_b200.losses wrappers"})
        if ext is not None:
            e2e.update({"extend_api_value": ext["value"], "extend_api_inserts_per_s": ext["inserts_per_s"],
                        "extend_api_extend_ms": ext["extend_ms"], "extend_api_h2d_bytes_per_step": ext["h2d_bytes_per_step"],
                        "extend_api_d2h_bytes_per_step": ext["d2h_bytes_per_step"], "extend_api_phase_us": ext["timing"],
                        "extend_api_path": "the drop-in shape of Trainer.step: ReplayDataset.extend(1280 reference tuples = lz4 blocks of concat(st, st_next), "
                                           "agent.py:78-81) -- compressed bytes over PCIe, LZ4 decode + de-duplication on the device (K6), K2b marks + K1 -- "
                                           "then the same CUDA-graph replay of the L batches and the double-buffered result read-back; 640 sampled per "
                                           "1280 inserted transitions at batch 32, as the reference's own step does"})
        line = {
            "metric": METRIC, "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(secs / args.steps * 1e3, 5), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8 frames / f32 targets / f64 n-step returns",
            "data": "synthetic",
            "config": shared_config(wl, L, A, ring, args),
            "timing": dict(timing, note=f"one block of exactly --steps {args.steps} steps after {SETTLE} + --warmup {args.warmup} untimed steps"),
            "timed_region_s": timing["timed_region_s"],
            "run": {"frame_ring_GB_per_gpu": round((ring * 1.0625 + 65536) * F_BYTES / 1e9, 2), "cuda_graph": not args.no_graph,
                    "uniforms": "torch uniform_ launch" if RNG_SEED is None else "Philox4x32-10 inside K2a (a0_pt_sample_rng)",
                    "gather_waves_batches": wave_sizes, "gather_window_draws": wave_window,
                    "k4_stream": "high-priority stream of the loop" if (wave_sizes and K4_PRIORITY) else "caller's stream",
                    "sharding": f"{world} independent shards, no data-path collective", "fill_seconds": round(t_fill, 1)},
            "clocks": clk.summary(),
            "e2e": e2e,
            "gpu_launches": launches_per_step * args.steps * len(blocks),
            "roofline": roofline,
            "cpu_baseline": cpu,
            "configs": configs,
            "learner_scaling": learner,
            "extra": extra,
        }
        EMIT(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def learner_scaling(args, torch, dist, world, rank, barrier, reduce_max, A, algo="c51", B=512, L=20, ring=200_000):
    """configs[4]: sharded PER replay + DATA-PARALLEL LEARNER, the gradient all-reduce INSIDE the timed region.
    One learner update = draw + gather (K2a, K3-f32) -> Nature-CNN forward (online, target, double-Q selection) -> K4 ->
    backward from the kernel's gradient -> NCCL all-reduce(SUM) of the flat gradient buffer, issued bucket by bucket
    from backward hooks (dist.OverlappedGradBucket: 6.9 MB under the convolution backward, 0.3 MB exposed) -> Adam ->
    K2b; L = 20 updates per Trainer.learn() replayed as one CUDA graph, per-GPU batch fixed (weak scaling).  The same
    loop is timed a second time with the collectives switched off: the difference is the exposed all-reduce time."""
    from agent0_b200.config import make_config
    from agent0_b200.synth import fill_shard_synthetic
    from agent0_b200.trainer import Trainer
    pg = dist.group.WORLD if world > 1 else None
    out = {"algo": algo, "batch_per_gpu": B, "global_batch": B * world, "updates_per_learn": L, "n_gpus": world,
           "ring_per_gpu": ring}

    def build(exchange, graph, amp=False):
        cfg = make_config(algo, per=True, n_step=3, batch_size=B, double_q=True, dueling=True, replay_size=ring, num_envs=16,
                          action_dim=A)
        cfg.learner.learner_steps = L
        cfg.learner.target_update_freq = 500
        tr = Trainer(cfg, process_group=pg, native_nstep=True, graph=graph, fused_input=True, sampler_seed=4242 + rank, amp=amp)
        if world > 1:
            tr.learner.bucket.enabled = exchange
        fill_shard_synthetic(tr.replay, ring, 16, 77 + rank)
        return tr

    def timed(tr, calls=4, blocks=3):
        for _ in range(3):
            tr.learn()
        torch.cuda.synchronize()
        ts = []
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(blocks):
            barrier()
            e0.record()
            for _ in range(calls):
                tr.learn()
            e1.record()
            torch.cuda.synchronize()
            barrier()
            ts.append(reduce_max(e0.elapsed_time(e1) / 1e3))
        return float(np.median(ts)) / (calls * L)

    graph = not args.no_graph
    try:
        tr = build(True, graph)
        sec = timed(tr)
    except Exception as e:
        if not graph:
            raise
        out["graph_capture_error"] = repr(e)[:300]
        graph = False
        torch.cuda.synchronize()
        tr = build(True, False)
        sec = timed(tr)
    out.update({"cuda_graph": graph, "ms_per_update": round(sec * 1e3, 4), "value": round(B * world / sec, 1), "unit": "transitions/s through the learner (CNN included)"})
    if world > 1:
        # the replicas took the same steps: the bit patterns of all parameters sum to the same integer on every rank
        bits = torch.cat([p.detach().reshape(-1) for p in tr.learner.model.parameters()]).view(torch.int32).long().sum().reshape(1)
        lo, hi = bits.clone(), bits.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        out["replicas_bit_identical"] = bool(lo.item() == hi.item())
        out["updates_taken"] = int(tr.learner.update_steps)
        bk = tr.learner.bucket
        out["allreduce_buckets_bytes"] = [int(hi - lo) * 4 for _, _, lo, hi in bk.buckets]
        del tr
        torch.cuda.empty_cache()
        tr2 = build(False, graph)
        sec0 = timed(tr2)
        out["ms_per_update_without_allreduce"] = round(sec0 * 1e3, 4)
        out["exposed_allreduce_us_per_update"] = round((sec - sec0) * 1e6, 2)
        del tr2
    else:
        del tr
    torch.cuda.empty_cache()
    try:        # the opt-in mixed-precision learner (bf16 gather + bf16 autocast, channels-last; fp32 weights, K4, Adam): not the reference's arithmetic
        tr3 = build(True, graph, amp=True)
        sec3 = timed(tr3)
        out["bf16_channels_last_ms_per_update"] = round(sec3 * 1e3, 4)
        out["bf16_channels_last_value"] = round(B * world / sec3, 1)
        del tr3
    except Exception as e:
        out["bf16_channels_last_error"] = repr(e)[:300]
    torch.cuda.empty_cache()
    return out


def hp_launches(wl, L):
    return 2 + L + (1 if wl["per"] else 0)


def grad_allreduce_probe(torch, dist, world, barrier, L):
    """The learner's only exchange step (SURVEY 8e) timed alone: one SUM all-reduce of the flat gradient bucket
    (C51 dueling: 1 814 943 fp32 parameters).  The learner-step scaling with the all-reduce INSIDE the timed
    region is the learner_* workloads' job (--workload learner_c51_b512)."""
    bucket = torch.zeros(1_814_943, dtype=torch.float32, device="cuda")
    for _ in range(5):
        dist.all_reduce(bucket)
    torch.cuda.synchronize(); barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(50):
        dist.all_reduce(bucket)
    e1.record(); torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / 50 * 1e3], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    us = float(t.item())
    return {"bytes": bucket.numel() * 4, "us_per_call": round(us, 2),
            "bus_GBps": round(2 * (world - 1) / world * bucket.numel() * 4 / (us * 1e-6) / 1e9, 1),
            "per_step_us_if_not_overlapped": round(us * L, 1)}


def weight_broadcast_probe(torch, dist, world, barrier, A):
    """SURVEY 8f-3 on hardware: the learner's weights handed to the other ranks (where on-box actors hold their copy of the
    net) with ONE flat NCCL broadcast (actor.broadcast_model) instead of a pickled state_dict per actor call
    (agent0/deepq/launch.py:33-36,56-61).  C51 dueling net, device time, max over ranks."""
    from agent0_b200.actor import broadcast_model
    from agent0_b200.config import make_config
    from agent0_b200.model import DeepQNet
    model = DeepQNet(make_config("c51", dueling=True, action_dim=A)).cuda()
    sent = 0
    for _ in range(3):
        sent = broadcast_model(model, src=0, process_group=dist.group.WORLD)
    torch.cuda.synchronize(); barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(20):
        broadcast_model(model, src=0, process_group=dist.group.WORLD)
    e1.record(); torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / 20 * 1e3], device="cuda", dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    us = float(t.item())
    return {"bytes": int(sent), "us_per_broadcast": round(us, 1), "GBps": round(sent / (us * 1e-6) / 1e9, 1),
            "note": "pack (torch.cat) + one NCCL broadcast + unpack in place; the reference pickles a state_dict over courier RPC per actor call"}


def time_workload(rp, name, args, torch, peak, L, A):
    """One BASELINE config on an existing shard: the step as a graph (median of blocks), K3 roofline, K4/K2 launch times."""
    wl = WORKLOADS[name]
    hp = HotPath(rp, wl, L, A, torch, variant=args.variant)
    bl = []
    secs = time_graphed(hp, 20, 5, torch, not args.no_graph, lambda: None, min_seconds=min(args.min_seconds, 0.15), stats=bl)
    secs_fused = time_graphed(hp, 20, 5, torch, not args.no_graph, lambda: None, step_fn=hp.step_fused_k4, min_seconds=0.02)
    secs_one = None
    if hp.waves:         # the same step with ONE gather launch in front of the first K4 (the round-1/2 schedule)
        hp1 = HotPath(rp, wl, L, A, torch, variant=args.variant, waves="none")
        secs_one = time_graphed(hp1, 20, 5, torch, not args.no_graph, lambda: None, min_seconds=0.03)
        del hp1
    hp.draw_pool()
    k4 = time_kernel(lambda i: hp.loss_k(i % L), 100, torch)
    k3 = time_kernel(lambda i: hp.gather(pool=i), 60, torch)
    k2a = time_kernel(lambda i: hp.sample(), 60, torch)
    k2b = time_kernel(lambda i: hp.update(), 60, torch) if wl["per"] else 0.0
    gb = bytes_per_transition(wl["n"]) * hp.total / k3 / 1e9
    full = {"transitions_per_s": round(hp.total * 20 / secs, 1), "ms_per_step": round(secs / 20 * 1e3, 4),
            "transitions_per_s_one_k4_launch_for_all_batches": round(hp.total * 20 / secs_fused, 1),
            "k4_us_per_batch": round(k4 * 1e6, 2), "k3_us": round(k3 * 1e6, 2), "k3_GBps": round(gb, 1),
            "k2a_us": round(k2a * 1e6, 2), "k2b_us": round(k2b * 1e6, 2), "desc": wl["desc"], "blocks": len(bl),
            "gather_waves_batches": [w[1] for w in hp.waves] if hp.waves else None,
            "transitions_per_s_single_gather_launch": round(hp.total * 20 / secs_one, 1) if secs_one else None,
            "step_GBps": round(bytes_per_transition(wl["n"]) * hp.total * 20 / secs / 1e9, 1)}
    compact = {"workload": name, "desc": wl["desc"], "value": full["transitions_per_s"], "ms_per_step": full["ms_per_step"],
               "k3_frac": round(gb / peak, 4), "k4_us": full["k4_us_per_batch"], "ring": rp.size}
    del hp
    return full, compact


def extras(rp, args, torch, peak, configs, entries):
    """Secondary numbers on the headline shard: the batch-512 configs that share it, K3 GB/s by launch size, the fused
    f32 gather, K1 and K6 as kernels."""
    out = {"workloads": {}, "k3_sweep": []}
    L, A = args.learner_steps, args.actions
    for name in ("c51_b512", "qr_b512", "iqn_b512"):
        full, compact = time_workload(rp, name, args, torch, peak, L, A)
        out["workloads"][name] = full
        configs.append(compact)
    # the headline workload with ONE gather launch in front of the first K4 (the schedule of rounds 1-2), for comparison
    try:
        wl = WORKLOADS[args.workload]
        hp1 = HotPath(rp, wl, L, A, torch, variant=args.variant, waves="none")
        s1 = time_graphed(hp1, 20, 5, torch, not args.no_graph, lambda: None, min_seconds=0.05)
        out["single_gather_launch"] = {"workload": args.workload, "transitions_per_s": round(hp1.total * 20 / s1, 1),
                                       "ms_per_step": round(s1 / 20 * 1e3, 5),
                                       "note": "gather_waves=None: K2a + one K3 launch complete before the first K4 starts"}
        del hp1
    except Exception as e:
        out["single_gather_launch"] = {"error": repr(e)[:300]}
    # the opt-in schedule that takes K2b off the critical path (hotloop.StaleByOneLoop): step s+1 draws while step s's
    # priorities are written back, i.e. with priorities one step stale -- the reference's prefetch queue does the same
    try:
        from agent0_b200.hotloop import StaleByOneLoop
        wl = WORKLOADS[args.workload]
        sl = StaleByOneLoop(rp, wl["algo"], wl["B"], L, A, net_outputs(wl["algo"], L * wl["B"], A, torch, rp.device), n_step=wl["n"],
                            double_q=wl["double"], per=wl["per"], discount=0.99, rng_seed=RNG_SEED)
        sl.capture()
        for _ in range(10):
            sl.run(publish=False)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        bl = []
        while sum(bl) < 0.1:
            e0.record()
            for _ in range(20):
                sl.run(publish=False)
            e1.record()
            torch.cuda.synchronize()
            bl.append(e0.elapsed_time(e1) / 1e3)
        sl.flush()
        med = float(np.median(bl))
        out["stale_by_one_schedule"] = {"workload": args.workload, "transitions_per_s": round(sl.total * 20 / med, 1),
                                        "ms_per_step": round(med / 20 * 1e3, 5), "blocks": len(bl),
                                        "note": "opt-in: K2b(s) on a side stream under K2a + K3 of step s+1 (priorities one step stale, as the "
                                                "reference's 3-deep prefetch); not the headline semantics"}
        del sl
    except Exception as e:      # measurement only
        out["stale_by_one_schedule"] = {"error": repr(e)[:300]}
    # K3 with the learner's input conversion fused in (a0_rb_gather_f32) against the three-pass
    # alternative it replaces: K3 to u8, then torch's .float() and .div(255) (agent.py:129-135)
    out["k3_f32"] = []
    from agent0_b200 import _lib as LB
    lib = LB.load()
    for name, count in (("c51_b32", 640), ("c51_b512", 10240)):
        wl = WORKLOADS[name]
        hp = HotPath(rp, wl, L, A, torch, variant=args.variant)
        hp.draw_pool()
        nbuf = 4 if count <= 1024 else 1
        obs = torch.empty(nbuf, count, 4 * F_BYTES, dtype=torch.float32, device=hp.dev)
        nxt = torch.empty_like(obs)

        def fused(i):
            LB.check(lib.a0_rb_gather_f32(rp.h, hp.idx_pool[i % INNER].data_ptr(), count, hp.n, 0.99, obs[i % nbuf].data_ptr(),
                                          nxt[i % nbuf].data_ptr(), 1, hp.act.data_ptr(), hp.r64.data_ptr(), hp.r32.data_ptr(),
                                          hp.d8.data_ptr(), hp.d32.data_ptr(), hp.boot.data_ptr(), hp._st()), "a0_rb_gather_f32")

        def three_pass(i):
            hp.gather(pool=i)
            x = hp.frames_pool[i % hp.n_out].view(count, 8, 84, 84).float().div(255.0)
            return x

        t_f = time_kernel(fused, 40, torch)
        t_3 = time_kernel(three_pass, 40, torch)
        by = (4 + min(wl["n"], 4)) * F_BYTES + 8 * F_BYTES * 4
        out["k3_f32"].append({"transitions": count, "fused_us": round(t_f * 1e6, 2), "three_pass_us": round(t_3 * 1e6, 2),
                              "fused_GBps": round(by * count / t_f / 1e9, 1), "frac_of_measured_peak": round(by * count / t_f / 1e9 / peak, 4),
                              "bytes_per_transition": by})
        del hp, obs, nxt
    # K1 as a kernel: a bulk append of 65 536 staged frames (device-resident staging, as the shard fill does):
    # F read + F written per frame
    try:
        nfr = 65536
        stage = torch.randint(0, 256, (nfr, F_BYTES), dtype=torch.uint8, device=rp.device)
        pos = (torch.randperm(rp.index.NF, device=rp.device)[:nfr]).to(torch.int32).contiguous()

        def k1(i):
            LB.check(lib.a0_rb_append(rp.h, stage.data_ptr(), pos.data_ptr(), nfr, None, 0, LB.stream_ptr(rp.device)), "a0_rb_append")
        t1 = time_kernel(k1, 40, torch)
        out["k1_roofline"] = {"kernel": "a0_k1_append", "frames_per_launch": nfr, "bytes_per_launch": 2 * nfr * F_BYTES,
                              "launch_us": round(t1 * 1e6, 2), "achieved_GBps": round(2 * nfr * F_BYTES / t1 / 1e9, 1),
                              "frac_of_measured_peak": round(2 * nfr * F_BYTES / t1 / 1e9 / peak, 4),
                              "note": "scattered ring slots; the staged frames were just read by the previous launch, so part of the read side hits L2"}
        del stage, pos
    except Exception as e:      # measurement only
        out["k1_roofline"] = {"error": repr(e)}
    # the drop-in ingest alone: ReplayDataset.extend with what the reference actor ships per Trainer.step
    try:
        from agent0_b200.config import make_config
        from agent0_b200.replay import ReplayDataset
        rq = ReplayDataset(make_config("c51", per=True, n_step=3, batch_size=32, replay_size=100_000, num_envs=16))
        rq.extend(entries[:1280])
        ms, tm = [], None
        for rep_ in range(3):
            for i in (1, 2, 3, 4):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                rq.extend(entries[i * 1280:(i + 1) * 1280])
                torch.cuda.synchronize()
                ms.append(round((time.perf_counter() - t0) * 1e3, 3))
                tm = rq.extend_timing()
        blob = float(np.mean([len(e[0]) for e in entries]))
        out["compat_extend"] = {"transitions": 1280, "ms": float(np.median(ms)), "ms_min": min(ms), "ms_all_calls": ms, "mean_blob_bytes": round(blob, 1),
                                "phase_us_last_call": tm,
                                "k6_decode_label": {"device_us": tm["device_decode_label_us"], "decoded_bytes": 1280 * 8 * F_BYTES,
                                                    "decoded_GBps": round(1280 * 8 * F_BYTES / (tm["device_decode_label_us"] * 1e-6) / 1e9, 1),
                                                    "bound": "one warp's dependent instruction chain per entry (LZ4 sequences are serial); not HBM"},
                                "note": "one a0_ex_extend call: compressed bytes staged + copied, K6 LZ4 decode + labels on the device, 8 label bytes "
                                        "per entry read back, host resolve + plan, K2b marks + K1 from the decoded scratch"}
        del rq
    except Exception as e:          # measurement only
        out["compat_extend"] = {"error": repr(e)}
    wl = dict(WORKLOADS["c51_b512"])
    hp = HotPath(rp, wl, 128, A, torch)           # buffers for up to 65536 transitions
    hp.draw_pool()
    for count in (32, 512, 640, 4096, 10240, 65536):
        for variant in (0, 3, 2, 1):
            dt = time_kernel(lambda i: hp.gather(count=count, variant=variant, pool=i), 40, torch)
            gb = bytes_per_transition(3) * count / dt / 1e9
            out["k3_sweep"].append({"transitions": count, "variant": ["tma_ring4", "ldg", "tma_full8", "tma_split2"][variant], "us": round(dt * 1e6, 2),
                                    "GBps": round(gb, 1), "frac_of_measured_peak": round(gb / peak, 4)})
    del hp
    return out


def extras_other_shards(args, torch, peak, configs):
    """The configs that need their own shard: configs[3] (FQF, M-DQN on a 2 M-transition shard) and configs[0]
    (DQN, uniform replay, n_step = 1) -- built after the headline shard has been released."""
    L, A = args.learner_steps, args.actions
    for names, ring in ((("fqf_b512", "mdqn_b512"), 2_000_000), (("dqn_b32_uniform",), 1_000_000)):
        try:
            rp, _ = make_shard(WORKLOADS[names[0]], ring, A, 0, torch, args.variant)
            for name in names:
                _, compact = time_workload(rp, name, args, torch, peak, L, A)
                configs.append(compact)
            del rp
            torch.cuda.empty_cache()
        except Exception as e:      # measurement only
            configs.append({"workload": names[0], "error": repr(e)})


# ------------------------------------------------------------------------------------------ CPU arm
def cpu_entries_for(wl, args):
    """The distinct lz4 tuples behind the CPU arm's deque (Actor.sample's packing, agent.py:64-81)."""
    from agent0_b200.synth import record_stream
    from oracle import cpu_path as CP
    E = 16
    s = record_stream(E, max(8, args.cpu_distinct // E) + wl["n"], seed=1234)
    tmp = CP.CpuReplay(args.cpu_distinct + 64, False)
    CP.fill_replay(tmp, s, wl["n"])
    return list(tmp.data)


def cpu_port(wl, L, A, args, entries):
    """oracle/cpu_path.py: the reference's pipeline restated, on a deque of args.cpu_entries entries."""
    import torch
    from oracle import cpu_path as CP
    B, algo = wl["B"], wl["algo"]
    rp = CP.CpuReplay(1_000_000, wl["per"])      # 1 M-slot priority vector as in the reference
    rep = -(-args.cpu_entries // len(entries))
    rp.extend((entries * rep)[:args.cpu_entries])
    o_all = net_outputs(algo, L * B, A, torch, "cpu")
    extra = dict(atoms=o_all.pop("atoms")) if algo == "c51" else {}
    if not (wl["double"] or algo in ("iqn", "fqf")):
        o_all["qsel"] = None
    outs = lambda it: {k: (v[it * B:(it + 1) * B].clone() if v is not None else None) for k, v in o_all.items()}
    gam = 0.99 ** wl["n"]
    return rp, (lambda fetch: CP.trainer_step(rp, fetch, outs, algo, L, gam, extra=extra))


def cpu_baseline(wl, L, A, args, workers):
    """The reference's host pipeline (oracle/cpu_path.py, single thread) on a bounded sample of the same workload."""
    import torch
    from oracle import cpu_path as CP
    cores = os.cpu_count() or 1
    torch.set_num_threads(1)
    entries = cpu_entries_for(wl, args)
    rp, mk = cpu_port(wl, L, A, args, entries)
    fetch, loader = CP.make_fetcher(rp, wl["B"], 0)
    step = lambda: mk(fetch)
    t0 = time.perf_counter(); step(); one = time.perf_counter() - t0
    steps = int(max(3, min(400, 12.0 / max(one, 1e-3))))      # ~12 s of CPU work
    n, dt = CP.time_steps(step, steps, 1)
    return {"value": round(n / dt, 1), "unit": UNIT, "cores": 1, "kind": "port", "host_cores_available": cores,
            "sample": f"{steps} Trainer.step loops x {L} batches x {wl['B']}, single thread, in-process fetch, on a "
                      f"{len(rp.data)}-entry lz4 deque ({len(entries)} distinct blobs) + torch CPU loss (1 intra-op thread); "
                      f"oracle/cpu_path.py; the all-cores run of the unmodified reference is `bench.py --impl reference`"}


def run_reference(args):
    """The reference arm: the UNMODIFIED reference (oracle/_ref, see oracle/ref_arm.py) through its own
    Trainer.step -- ReplayDataset, DataLoaderX(num_workers=2, pin_memory) + DataPrefetcher, learner.train, update_priority --
    with all host threads torch wants; the restated port (oracle/cpu_path.py) is timed beside it as a cross-check, and is
    the arm itself for the workloads whose networks the table stub does not cover (IQN, FQF) or when oracle/_ref is absent."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    L, A = args.learner_steps, args.actions
    cores = os.cpu_count() or 1
    import torch
    from oracle import cpu_path as CP
    from oracle import ref_arm as RA
    B, algo = wl["B"], wl["algo"]
    entries = cpu_entries_for(wl, args)
    steps = args.steps
    warm = max(1, min(args.warmup, 5))
    # ---- the port, all intra-op threads, in-process fetch and the reference's 2 workers: cross-check ----------------
    torch.set_num_threads(cores)
    rp, mk = cpu_port(wl, L, A, args, entries)
    port = {}
    for w in (0, 2):
        fetch, loader = CP.make_fetcher(rp, B, w)
        n, dt = CP.time_steps(lambda: mk(fetch), max(2, min(steps, 5)), 1)
        port[f"workers_{w}"] = round(n / dt, 1)
        del fetch, loader
    del rp, mk
    kind, v, ms, sample, used = "port", None, None, None, None
    if RA.available() and algo in RA.SUPPORTED:
        o = net_outputs(algo, L * B, A, torch, "cpu")
        if not wl["double"]:
            o["qsel"] = None
        tr = RA.make_trainer(algo, wl["per"], wl["n"], wl["double"], B, L, A, o, replay_size=1_000_000)
        n_entries = RA.fill(tr, entries, args.cpu_entries)
        for _ in range(warm):
            RA.step(tr)
        t0 = time.perf_counter()
        for _ in range(steps):
            RA.step(tr)
        dt = time.perf_counter() - t0
        v, ms, kind = round(L * B * steps / dt, 1), dt / steps * 1e3, "reference"
        used = min(cores, 2 + 1 + 1 + torch.get_num_threads())
        sample = (f"{steps} calls of the unmodified reference's Trainer.step (oracle/_ref, trainer.py:74-119): {L} x [DataLoaderX("
                  f"shuffle, num_workers=2, pin_memory={torch.cuda.is_available()}) + DataPrefetcher fetch of {B} entries from a {n_entries}-entry "
                  f"lz4 deque ({len(entries)} distinct blobs), .float(), IS weights over the 1 M-slot priority vector, {algo.upper()}Learner.train "
                  f"with table-lookup networks (CNN excluded on both arms), update_priority]; torch intra-op threads = {torch.get_num_threads()}; "
                  f"port cross-check (oracle/cpu_path.py, same deque): {port} transitions/s")
    else:
        best = max(port, key=port.get)
        w = int(best.split("_")[1])
        rp, mk = cpu_port(wl, L, A, args, entries)
        fetch, loader = CP.make_fetcher(rp, B, w)
        n, dt = CP.time_steps(lambda: mk(fetch), steps, warm)
        v, ms = round(n / dt, 1), dt / steps * 1e3
        used = min(cores, max(torch.get_num_threads(), w + 1))
        why = "oracle/_ref is absent" if not RA.available() else f"the table-network stub does not cover {algo}"
        sample = (f"{steps} Trainer.step loops x {L} batches x {B} through the restated pipeline (oracle/cpu_path.py; {why}) with "
                  f"{'in-process fetch' if w == 0 else str(w) + ' DataLoader workers'} on a {len(rp.data)}-entry lz4 deque; calibration {port}")
    EMIT(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": args.warmup, "ms_per_step": round(ms, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8 frames / f32 targets / f64 n-step returns", "data": "synthetic",
        "config": shared_config(wl, L, A, args.total_ring // max(1, args.gpus) if args.total_ring else args.ring, args),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": used, "host_cores_available": cores, "kind": kind, "sample": sample,
                         "port_crosscheck": port},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def _json_only_stdout():
    """Everything any library prints to stdout while the benchmark runs (NCCL's version banner, for
    one) goes to stderr; the process's real stdout receives exactly the one JSON line."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    out = os.fdopen(real, "w")
    sys.stdout = sys.stderr

    def emit(line):
        out.write(line + "\n")
        out.flush()
    return emit


if __name__ == "__main__":
    a = parse()
    EMIT = _json_only_stdout()
    if a.impl == "reference":
        run_reference(a)
        # The reference's pump leaves daemon threads behind (BackgroundGenerator, the DataLoader's pin-memory thread and
        # worker processes: utils.py:45-61); tearing the interpreter down under them intermittently ends in
        # "terminate called without an active exception" (exit code 134) AFTER the line has been printed.  The line is out
        # and flushed: leave without running the teardown.
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)
    else:
        run_ours(a)
