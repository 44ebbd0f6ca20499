"""The step the benchmark times -- hotloop.ReplayTargetLoop captured into a CUDA graph and replayed (the mailbox sampler,
the gather in waves on a side stream with the ordered-fetch window, K4 on the high-priority stream joined at the waves
with PDL, C51's early links, the planned or overlapped write-back, top / beta and the sampler's call counter resident on
the device) -- against a lockstep CPU reference of the whole step, replay after replay.

The reference is assembled from oracles that are pinned on their own and shares no kernel with the loop:
  ingest      agent0_b200.ring_index.RingIndex (the index's specification) fed the same steps, its marks applied to an
              oracle SumTree (a new leaf is max_p^alpha, an evicted one 0), an owner map from ring position to
              (stream, step), beta from oracle.reference_replay.LinearSchedule;
  draw        SumTree.sample on philox_uniform(seed, call) -- oracle/sample_unique.py for the draw without replacement --
              with the call number the replay must use; IS weights in float64 (trainer.py:91-94);
  gather      the stacks and n-step scalars of oracle.reference_replay.pack_nstep through the owner map;
  targets     oracle/losses64.py on the network outputs and the reference's gathered scalars: the per-element bound
              (n + 16) 2^-24 s64 and the 1e-5 contract (tests/parity.py);
  write-back  SumTree.update with the device's losses (they are only within tolerance of the reference: a one-ulp
              difference would fork every later draw).
Every stage is checked before the next one uses it, and the next replay draws from the reference tree just checked, so
an error that every schedule of the loop shares -- a K4 that reads a wave before its wait, a write-back that races the
next draw, a scalar published one replay late, a call counter advanced twice -- fails here where a comparison of one
schedule with another cannot see it.  Output buffers are poisoned before every step: an element no kernel wrote fails."""
import functools
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import torch

from bench import WORKLOADS, net_outputs
from oracle import losses64 as O64
from oracle import reference_replay as OR
from oracle.sample_unique import sample_unique
from oracle.sumtree import SumTree, new_priority, philox_uniform
from tests import parity
from tests.test_gpu_edges import _stream
from tests.test_gpu_loss_shapes import TINY, _quantile_refs
from tests.test_gpu_tree_depths import _is_weights

f32 = np.float32
E, N, A, HW = 16, 8192, 4, (84, 84)           # 2^13 leaves: deeper than the sampler's 10-level shared-memory top
FILL = 640                                   # steps before the first step: 10 240 records through 8192 slots
REPLAYS = 3                                  # captured replays per case, after the eager step of the warm-up
STEPS = FILL + REPLAYS
GAMMA = 0.99
TOTAL_STEPS = 2 * N                          # a short beta schedule: beta moves by 6e-4 with every step's ingest
SEED = 20261017                              # the sampler's Philox seed (bench.py's)
CALL0 = 1000                                 # the call number of the eager step; replay i uses CALL0 + 1 + i

# name -> (algo, B, L, per, n, double, loop options)
CASES = {name: (w["algo"], w["B"], 20, w["per"], w["n"], w["double"], {}) for name, w in WORKLOADS.items()}
CASES.update({
    # 1024 draws: the planned write-back (a0_pt_update_plan / _apply); 1025: the chunk schedule under the last K4
    "dqn_64x16": ("dqn", 64, 16, True, 3, True, {}), "dqn_41x25": ("dqn", 41, 25, True, 3, True, {}),
    "iqn_64x16": ("iqn", 64, 16, True, 3, True, {}), "iqn_41x25": ("iqn", 41, 25, True, 3, True, {}),
    # a batch's gather moves 9.93 MB (doubling waves) and 10.05 MB (one wave per batch); 89 is not a multiple of 4
    "c51_88x5": ("c51", 88, 5, True, 3, True, {}), "c51_89x5": ("c51", 89, 5, True, 3, True, {}),
    "mdqn_L1": ("mdqn", 32, 1, True, 3, False, {}),            # no waves
    "fqf_L2": ("fqf", 32, 2, True, 3, True, {}),               # waves, no plan join (_plan_join == L)
    "qr_B1": ("qr", 1, 20, True, 3, True, {}),                 # single-draw batches: the last-CTA weight epilogue
    "c51_waves_plain_joins": ("c51", 32, 20, True, 3, True,    # the join path that switches PDL off and on again
                              dict(gather_waves=[1, 2, 3, 6, 8], pdl_at_joins=False, gather_window=1, k4_priority=False)),
    "c51_unique": ("c51", 32, 20, True, 3, True, dict(replacement=False)),
})


@functools.lru_cache(maxsize=1)
def stream():
    """E host streams of STEPS steps: 84x84 frames, whole new stacks (p = 0.1) and static screens (p = 0.05), fractional
    float64 rewards, terminal steps with p = 0.15, actions below A."""
    obs, n_new, act, rew, done = _stream(E, STEPS, HW, seed=17, p_new4=0.1, p_static=0.05)
    return obs, n_new, act % A, rew, done


@functools.lru_cache(maxsize=2)
def nstep_scalars(n):
    """Action, n-step return and done of every entry (k * E + e) of pack_nstep: the scalars do not depend on the frames,
    so it runs on one-byte stand-ins for the stacks."""
    obs, _, act, rew, done = stream()
    _, a, r, d = OR.pack_nstep(np.zeros((STEPS + 1, E, 1), np.uint8), act, rew, done, n, GAMMA)
    return a, r, d


def entry_frames(obs, e, j, n):
    """pack_nstep's frames of stream e's record j, concat(st, st_next) = concat(obs[j], obs[j + n]) (its entry is
    (j + n - 1) * E + e), for arrays of records."""
    return np.concatenate((obs[j, e], obs[j + n, e]), axis=1).reshape(len(j), -1)


def test_entry_frames_restate_pack_nstep():
    """The reference gathers frames record by record instead of materialising every entry of the stream (300 MB per
    entry set here): the restatement must be pack_nstep's frames, and nstep_scalars its other columns."""
    for n in (1, 3):
        Es, T = 3, 12
        obs, _, act, rew, done = _stream(Es, T, (4, 4), seed=n, p_new4=0.2, p_static=0.2)
        fr, a, r, d = OR.pack_nstep(obs, act, rew, done, n, GAMMA)
        _, a1, r1, d1 = OR.pack_nstep(np.zeros((T + 1, Es, 1), np.uint8), act, rew, done, n, GAMMA)
        assert np.array_equal(a, a1) and np.array_equal(r.view(np.int64), r1.view(np.int64)) and np.array_equal(d, d1)
        j, e = np.divmod(np.arange((T - n + 1) * Es), Es)
        assert np.array_equal(entry_frames(obs, e, j, n), fr[(j + n - 1) * Es + e])


def _bits_equal(name, got, want):
    g, w = np.ascontiguousarray(got), np.ascontiguousarray(want)
    assert g.shape == w.shape, f"{name}: shape {g.shape} vs {w.shape}"
    bad = np.flatnonzero(g.reshape(-1).view(f"u{g.itemsize}") != w.reshape(-1).view(f"u{w.itemsize}"))
    assert bad.size == 0, f"{name}: {bad.size} elements differ, first at {bad[:6].tolist()}: {g.reshape(-1)[bad[:3]]} vs {w.reshape(-1)[bad[:3]]}"


class StepReference:
    """The shard, driven from the host stream, and its lockstep reference (module docstring)."""

    def __init__(self, algo, per, n, B, replacement):
        from agent0_b200.config import make_config
        from agent0_b200.replay import ReplayDataset
        from agent0_b200.ring_index import RingIndex
        self.algo, self.per, self.n, self.B, self.replacement = algo, per, n, B, replacement
        cfg = make_config(algo, per=per, n_step=n, batch_size=B, replay_size=N, double_q=True, dueling=True, num_envs=E,
                          action_dim=A)
        cfg.trainer.total_steps = TOTAL_STEPS
        cfg.learner.discount = GAMMA
        self.rp = rp = ReplayDataset(cfg, native_nstep=True)
        self.P = rp.P
        self.spec = RingIndex(N, rp.index.NF, n, rp.index.age_limit)
        self.tree = SumTree(N)
        assert self.tree.P == self.P
        self.alpha = 0.5 if per else 0.0                    # the shard's: a uniform shard marks max_p^0 = 1
        assert rp.alpha == self.alpha
        self.max_p = f32(1.0)
        self.beta_schedule = OR.LinearSchedule(0.4, 1.0, TOTAL_STEPS) if per else None
        self.beta = 0.4 if per else 1.0
        self.own_e = np.full(N, -1, np.int64)                # ring position -> (stream, step) of the record it holds
        self.own_j = np.full(N, -1, np.int64)
        self.own_q = np.full(N, -1, np.int64)                # ... and its record sequence number (>= N: the ring wrapped)
        self.steps = 0
        self.seen_wrapped = self.seen_terminal = False      # negative controls, over the draws of the case
        obs = stream()[0]
        z = np.zeros(0, np.int64)
        self.spec.plan(z, np.zeros((0, 8), np.int64), np.arange(4 * E), z, z.astype(np.float64), z.astype(bool))
        self.last4 = {e: np.arange(4 * e, 4 * e + 4, dtype=np.int64) for e in range(E)}
        rp.reset_streams(np.arange(E), obs[0])
        assert float(rp.max_p_tensor) == 1.0
        for _ in range(FILL):
            self.ingest()
        assert self.spec.head_q > N and self.spec.tail_q > 0            # the ring wrapped, records were evicted
        self.check_ingest()
        self.lib = rp.lib

    # ------------------------------------------------------------------------------------------------ ingest
    def ingest(self, publish_dynamic=False):
        obs, n_new, act, rew, done = stream()
        k, es = self.steps, np.arange(E)
        new = [obs[k + 1][e, 4 - n_new[k][e]:] for e in es if n_new[k][e]]
        new = np.concatenate(new) if new else np.zeros((0,) + HW, np.uint8)
        self.rp.append_steps(es, n_new[k], new, act[k], rew[k], done[k], publish_dynamic=publish_dynamic)
        fs8 = self.spec.resolve_shift(es, n_new[k], self.last4)
        q0 = self.spec.head_q
        marks = self.spec.plan(es, fs8, np.arange(int(n_new[k].sum())), act[k], rew[k], done[k]).marks
        q = q0 + es
        self.own_e[q % N], self.own_j[q % N], self.own_q[q % N] = es, k, q
        if marks.size:                              # in order: evictions, then the records that became sampleable
            pos = np.where(marks >= 0, marks, ~marks)
            self.tree.set(pos, np.where(marks >= 0, new_priority(self.max_p, 0.0, self.alpha), f32(0)))
        if self.per:
            self.beta = self.beta_schedule(E)       # replay.py:53: the value before this ingest's advance
        self.steps += 1
        self.marks = marks

    def check_ingest(self):
        rp = self.rp
        torch.cuda.synchronize()
        tree = rp.tree.cpu().numpy()
        leaves = tree[self.P:self.P + N]
        assert np.array_equal(leaves > 0, self.spec.sampleable), "live leaves are not the specification's sampleable records"
        assert rp.index.top == self.spec.top and rp.beta == self.beta
        m = self.marks
        new = leaves[m[m >= 0]]
        assert (new == new_priority(self.max_p, 0.0, self.alpha)).all(), f"new leaves {new[:4]} != max_p^alpha of {self.max_p}"
        gone = ~m[m < 0]
        assert (leaves[gone[~self.spec.sampleable[gone]]] == 0).all(), "an evicted leaf is not 0"
        ref = SumTree(N)
        ref.build(leaves)
        _bits_equal("tree after the ingest vs SumTree.build of its leaves", tree, ref.nodes)
        _bits_equal("tree after the ingest vs the reference", tree, self.tree.nodes)

    # ------------------------------------------------------------------------------------------------ one step
    def check_step(self, loop, call, on, tag):
        """Draw, gather, targets, write-back and fault word of the step that just ran with sampler call ``call``."""
        torch.cuda.synchronize()
        B, L, T, n = loop.B, loop.L, loop.total, self.n
        top = self.spec.top
        beta = self.beta
        root = self.tree.root
        # ---- draw
        if self.replacement:
            r_idx, r_prio = self.tree.sample(philox_uniform(SEED, call, T), B)
            other = self.tree.sample(philox_uniform(SEED, call + 1, T), B)[0]
        else:
            r_idx, r_prio, _, _, short = sample_unique(self.tree.nodes, self.P, SEED, call, L, B, top, beta, 0.0, not self.per)
            assert not short.any()
            other = sample_unique(self.tree.nodes, self.P, SEED, call + 1, L, B, top, beta, 0.0, not self.per)[0]
            assert all(len(set(r_idx[b * B:(b + 1) * B])) == B for b in range(L))
        idx = loop.idx.cpu().numpy()
        _bits_equal(f"{tag}: drawn indices", idx, r_idx)
        _bits_equal(f"{tag}: drawn priorities", loop.prio.cpu().numpy(), r_prio)
        assert not np.array_equal(other, r_idx), f"{tag}: call {call} + 1 draws the same indices: the call check is vacuous"
        w = loop.w.cpu().numpy()
        if self.per:
            parity.close(f"step.{self.algo}.is_weights", w, _is_weights(r_prio, root, top, beta, 0.0, B))
        else:
            assert (w == 1.0).all(), f"{tag}: a uniform draw's IS weights must be exactly 1"
        # ---- gather
        obs = stream()[0]
        a_ref, r_ref, d_ref = nstep_scalars(n)
        e, j = self.own_e[idx], self.own_j[idx]
        ent = (j + n - 1) * E + e
        _bits_equal(f"{tag}: action", loop.act.cpu().numpy(), a_ref[ent])
        _bits_equal(f"{tag}: n-step return (f64)", loop.r64.cpu().numpy(), r_ref[ent])
        _bits_equal(f"{tag}: n-step return (f32)", loop.r32.cpu().numpy(), r_ref[ent].astype(f32))
        _bits_equal(f"{tag}: done (u8)", loop.d8.cpu().numpy(), d_ref[ent].astype(np.uint8))
        _bits_equal(f"{tag}: done (f32)", loop.d32.cpu().numpy(), d_ref[ent].astype(f32))
        boot = np.where(j + n < self.steps, ((j + n) * E + e) % N, -1)
        _bits_equal(f"{tag}: bootstrap index", loop.boot.cpu().numpy(), boot)
        for lo in range(0, T, 512):
            hi = min(T, lo + 512)
            _bits_equal(f"{tag}: stacks of draws [{lo}, {hi})", loop.frames[lo:hi].cpu().numpy(),
                        entry_frames(obs, e[lo:hi], j[lo:hi], n))
        self.seen_wrapped |= bool((self.own_q[idx] >= N).any())
        self.seen_terminal |= bool(d_ref[ent].any())
        # ---- targets: network outputs + the reference's gathered scalars (+ the device weights, checked above)
        got = {"loss": loop.loss.cpu().numpy(), "grad": loop.grad.cpu().numpy(), "prio": loop.newp.cpu().numpy()}
        if self.algo == "fqf":
            got.update(fraction_loss=loop.frac.cpu().numpy(), grad_taus=loop.gtau.cpu().numpy())
        a, r, d = a_ref[ent], r_ref[ent].astype(f32), d_ref[ent].astype(f32)
        rows = [slice(k * B, (k + 1) * B) for k in range(L)]
        # the float64 references of a batch-512 QR step are ~20 s of numpy on one core; the checks stay in this thread
        with ThreadPoolExecutor(max_workers=4) as ex:
            refs = ex.map(lambda s: target_refs(loop, on, s, a[s], r[s], d[s], w[s]), rows)
            for s, ref in zip(rows, refs):
                check_targets(f"step.{self.algo}", {key: v[s] for key, v in got.items()}, ref, s, loop)
        # ---- write-back, with the device's losses
        before = self.tree.nodes.copy()
        if self.per:
            self.max_p = self.tree.update(idx, got["loss"], loop.eps, loop.alpha, self.max_p)
            assert not np.array_equal(before, self.tree.nodes), f"{tag}: the write-back changed nothing"
        _bits_equal(f"{tag}: tree after the write-back", self.rp.tree.cpu().numpy(), self.tree.nodes)
        _bits_equal(f"{tag}: max_p", self.rp.max_p_tensor.cpu().numpy(), np.array([self.max_p], f32))
        assert self.lib.a0_rb_check_fault(self.rp.h) == 0, f"{tag}: fault word"
        return idx


def target_refs(loop, on, s, a, r, d, w):
    """The float64 value (losses64.R) of every output of batch rows ``s``, and the error scales of
    tests/test_gpu_loss_shapes.py where an output is a difference of larger operands."""
    algo, G = loop.algo, loop.gamma_n
    B = len(a)
    bi = np.arange(B)
    o = {k: (v if k == "atoms" else v[s]) for k, v in on.items()}
    qs = o["qsel"] if (loop.double_q or algo in ("iqn", "fqf")) and algo != "mdqn" else None
    scales = {}
    if algo in ("dqn", "mdqn"):
        # the gradient w * clamp(q - T) is a difference of operands of magnitude max(|q|, |T|)
        q, tn = o["online"], o["tgt_next"]
        sc = float(max(np.abs(q).max(), np.abs(tn).max() + np.abs(r).max() + 1.0) * w.max())
        if algo == "dqn":
            ref64 = O64.dqn(q, tn, qs, a, r, d, w, G)
            scales = {"grad": sc}
        else:
            tau, lo = loop.mdqn
            ref64 = O64.mdqn(q, tn, o["tgt_cur"], a, r, d, w, G, tau, lo)
            scales = {"loss": sc * sc / 2, "grad": sc}
    elif algo == "c51":
        M, vmin, vmax = loop.c51
        ref64 = O64.c51(o["online"], o["tgt_next"], qs, a, r, d, w, G, o["atoms"], vmin, vmax)
        # the gradient w * (p_j * sum(m) - m_j) is a difference of operands of size up to w
        wm = np.abs(w)[:, None] * ref64.pop("target_prob").v
        scales = {"grad": float((np.abs(ref64["grad"].v[bi, a] + wm) + wm).max())}
    elif algo == "qr":
        N_ = o["online"].shape[2]
        _, ref64, *_ = _quantile_refs(o["online"], o["tgt_next"], None, qs, a, r, d, w, G, 0, N_, N_, True)
    elif algo == "iqn":
        _, ref64, *_ = _quantile_refs(o["online"], o["tgt_next"], o["taus"], qs, a, r, d, w, G, 1,
                                      o["tgt_next"].shape[1], o["online"].shape[1], True)
    else:
        F = o["online"].shape[1]
        _, ref64, *_ = _quantile_refs(o["online"], o["tgt_next"], o["taus_hat"], qs, a, r, d, w, G, 1, F, F, True)
        ref64.update(O64.fraction(o["online"][bi, :, a], o["q_bar"][bi, :, a], o["taus"], w))
    return ref64, scales


def check_targets(name, got, refs, s, loop):
    """Every output of batch rows ``s`` against its float64 value: within (n + 16) 2^-24 s64 (an element with s64 = 0
    must be exactly 0) and within the 1e-5 contract (tests/parity.py); the priorities against the float64
    (loss + eps)^alpha.  (The fp32 oracle is no yardstick at 10 240 draws: its own rounding in a 200-term QR gradient
    sum is as large as the kernel's, and their difference reaches 1.05e-5.)"""
    ref64, scales = refs
    for k, ref in ref64.items():
        g = got[k].astype(np.float64)
        tol = (ref.n + 16) * 2.0 ** -24 * ref.s + np.where(ref.s > 0, TINY, 0.0)
        bad = ~(np.abs(g - ref.v) <= tol)
        assert not bad.any(), (f"{name}.{k}: {int(bad.sum())} elements outside the float64 bound, e.g. index "
                               f"{np.argwhere(bad)[0].tolist()} (rows {s.start}+): got {g[bad][0]!r}, float64 {ref.v[bad][0]!r}")
        parity.close(f"{name}.{k}", got[k], ref.v, scale=scales.get(k))
    parity.close(f"{name}.prio", got["prio"], O64.priority(got["loss"], loop.eps, loop.alpha))


def _poison(loop):
    """Every output of the step to a value no kernel writes, before the step."""
    nan = float("nan")
    for t in (loop.loss, loop.grad, loop.newp, loop.prio, loop.w, loop.r32, loop.d32, loop.r64) + \
            ((loop.frac, loop.gtau) if loop.algo == "fqf" else ()):
        t.fill_(nan)
    for t in (loop.idx, loop.act, loop.boot):
        t.fill_(-7)
    loop.d8.fill_(7)
    loop.frames.fill_(0x5A)


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(CASES))
def test_captured_step_equals_the_lockstep_reference(case):
    """One eager step (capture()'s warm-up: the single gather launch) and REPLAYS graph replays of the captured default
    schedule, with one step of every stream ingested before each replay -- alternately published by the ingest launch
    (append_steps(publish_dynamic=True) + run(publish=False), bench.py's e2e path) and by run()'s push_dynamic -- each
    checked stage by stage against the reference.  Negative controls: consecutive steps draw different batches, the tree
    and beta move from step to step, the draws include records of the wrapped ring and terminal records."""
    from agent0_b200.hotloop import ReplayTargetLoop
    algo, B, L, per, n, double, opts = CASES[case]
    replacement = opts.get("replacement", True)
    ref = StepReference(algo, per, n, B, replacement)
    rp = ref.rp
    o = net_outputs(algo, B * L, A, torch, rp.device)
    on = {k: v.cpu().numpy() for k, v in o.items()}
    loop = ReplayTargetLoop(rp, algo, B, L, A, o, n_step=n, double_q=double, per=per, discount=GAMMA, rng_seed=SEED,
                            want_prio=True, **opts)
    if case == "mdqn_L1" or not replacement:
        assert loop.waves is None
    elif case == "c51_89x5":
        assert [w[1] for w in loop.waves] == [1] * L and not loop._use_plan
    elif case == "c51_88x5":
        assert [w[1] for w in loop.waves] == [1, 1, 3] and loop._use_plan
    elif case == "fqf_L2":
        assert len(loop.waves) == 2 and loop._plan_join == L and not loop._use_plan
    elif case in ("dqn_64x16", "iqn_64x16", "c51_b32", "qr_B1"):
        assert loop._use_plan
    elif case in ("dqn_41x25", "iqn_41x25"):
        assert loop.waves and not loop._use_plan
    draws, trees, betas = [], [], []
    rp.rng_seek(CALL0)
    _poison(loop)
    loop.capture(warm=1)              # push_dynamic, one eager step with call CALL0, then the capture (nothing runs)
    draws.append(ref.check_step(loop, CALL0, on, f"{case} eager step"))
    trees.append(ref.tree.nodes.copy()); betas.append(ref.beta)
    for i in range(REPLAYS):
        dyn = i % 2 == 0
        ref.ingest(publish_dynamic=dyn)
        ref.check_ingest()
        _poison(loop)
        loop.run(publish=not dyn)
        draws.append(ref.check_step(loop, CALL0 + 1 + i, on, f"{case} replay {i}"))
        trees.append(ref.tree.nodes.copy()); betas.append(ref.beta)
    for s in range(1, len(draws)):
        assert not np.array_equal(draws[s], draws[s - 1]), f"steps {s - 1} and {s} drew the same batches"
        assert not np.array_equal(trees[s], trees[s - 1]) or not per, f"the tree did not change between steps {s - 1} and {s}"
    assert betas[0] != betas[-1] or not per
    assert ref.seen_wrapped and ref.seen_terminal, "the draws never reached a record of the wrapped ring or a terminal record"
