"""The inner loop of the reference's ``Trainer.step`` (agent0/deepq/trainer.py:82-104) as a pre-bound,
CUDA-graph-capturable sequence of C-ABI launches, for callers that supply the network outputs
themselves (a training loop owns the CNN; bench.py pre-generates them because the BASELINE metric
excludes the CNN).

Per ``step()``: draw L = learner_steps batches of B transitions (K2a, one launch), gather them (K3,
one launch: stack reconstruction + n-step return), run the fused target/loss kernel once per batch
(K4, L launches: in training every batch's outputs depend on the previous optimizer step, so they
stay separate launches), write the new priorities (K2b, one launch).  All buffers are allocated
once; every launch is a single ctypes call with pre-built argument blocks, so the host cost per
step is ~25 ctypes calls -- or one ``graph.replay()`` after ``capture()``.  ``sample(dynamic=True)``
semantics: top/beta are read from the device values published by ``ReplayDataset.push_dynamic``,
so a captured graph keeps following the shard as it grows and beta anneals.

The general-purpose wrappers (``ReplayDataset.sample``, ``agent0_b200.losses``) allocate their
outputs and validate their inputs on every call; this class is the same work without that.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib

ALGOS = ("dqn", "mdqn", "c51", "qr", "iqn", "fqf")


def wave_plan(L, B, frame_bytes, spec="auto"):
    """The gather waves of a draw of L batches of B transitions: [(first batch, batches, first draw, draws)] per wave, or
    None for a single gather launch.  spec "auto": one wave per batch when a batch's gather (16 frames of traffic per
    transition) moves 10 MB or more -- it then outlasts a K4 launch, and the target kernels hide under the following
    waves; otherwise the K4 chain is the longer side and the waves only have to stay ahead of it: 1, 1, 2, 4, ...
    batches (a tail shorter than its predecessor joins it).  A list gives the wave sizes in batches; None / 0 / a single
    wave / L < 2: no waves."""
    if not spec or L < 2:
        return None
    if isinstance(spec, str):
        assert spec == "auto", spec
        if B * 16 * frame_bytes >= 10_000_000:
            sizes = [1] * L
        else:
            sizes, w = [1], 1
            while sum(sizes) < L:
                sizes.append(min(w, L - sum(sizes)))
                w *= 2
            if len(sizes) > 1 and sizes[-1] < sizes[-2]:
                tail = sizes.pop()
                sizes[-1] += tail
    else:
        sizes = [int(x) for x in spec]
        assert all(x > 0 for x in sizes) and sum(sizes) == L, "gather_waves must be positive batch counts that sum to learner_steps"
    if len(sizes) < 2:
        return None
    plan, b0 = [], 0
    for n in sizes:
        plan.append((b0, n, b0 * B, n * B))
        b0 += n
    return plan


def early_links(L, waves, plan_join=None):
    """The K4 links of a waved step that may run their batch-side work before griddepcontrol.wait (a0_loss_c51_linked,
    A0_C51_EARLY): those whose sole predecessor is the previous K4.  A link launches once the link ahead of it has
    passed its own wait, so everything that link joined -- the wave that holds this batch, the draw before it -- is
    complete.  A link that itself joins a wave (the first batch of each) or the write-back plan (``plan_join``) has a
    second predecessor and reads nothing before its wait.  waves: wave_plan's rows; None (the single gather launch):
    no link."""
    if not waves:
        return frozenset()
    joins = {b0 for b0, _, _, _ in waves}
    if plan_join is not None:
        joins.add(plan_join)
    return frozenset(k for k in range(L) if k not in joins)


class ReplayTargetLoop:
    def __init__(self, replay, algo, batch_size, learner_steps, action_dim, outputs, n_step=None, double_q=True,
                 per=None, variant=0, discount=None, alpha=0.5, eps=0.01, c51=(51, -10.0, 10.0), mdqn=(0.03, -1.0),
                 frames=None, rng_seed=None, overlap_sample_gather=None, want_prio=False, early_update=True,
                 gather_waves="auto", pdl_at_joins=True, gather_window="auto", k4_priority=True, waves_when_eager=False,
                 replacement=True):
        """replay: ReplayDataset (native_nstep=True when n_step > 1).  outputs: dict of STATIC f32 device
        tensors holding the network outputs of all L*B sampled transitions, batch k in rows
        [k*B, (k+1)*B): ``online``, ``tgt_next`` (+ ``qsel`` [L*B,A] under double_q / for iqn, fqf;
        ``tgt_cur`` for mdqn; ``atoms`` [M] for c51; ``taus`` for iqn; ``taus``, ``taus_hat``, ``q_bar`` for
        fqf), shaped as the learners produce them (agent0_b200.losses).  frames: optional u8
        [L*B, 8*F] output buffer for the gather (allocated if None).  rng_seed: the sampler draws its own
        uniforms (Philox inside K2a, device-resident call counter advanced by every launch/replay)
        instead of reading ``self.u``, which ``step()`` otherwise refills with ``uniform_()``.
        want_prio: K4 also writes (loss+eps)^alpha per sample into ``self.newp`` (the loop itself does not need it:
        K2b recomputes the priority from the loss).
        overlap_sample_gather: ``step()`` issues K2a and K3 through a0_rb_sample_gather (the gather runs
        under the sampler, fed draw by draw through a mailbox) instead of back to back; same results.
        gather_waves: the gather of the L batches is cut into waves (a0_rb_sample_mail + one a0_rb_gather_mail per
        wave) on a side stream, and batch k's K4 waits only for the wave that holds batch k -- the later batches
        are fetched UNDER the target kernels of the earlier ones (what the reference's DataPrefetcher does with its
        3-deep queue, utils.py:45-61).  "auto": doubling waves of 1, 1, 2, 4 ... batches when a batch is small
        (the K4 chain is the longer side), one wave per batch when a batch moves more than ~10 MB; a list gives
        the wave sizes in batches; None/0: one gather launch on the caller's stream.  Same results either way.
        gather_window: ordered fetch inside the waves (a0_rb_gather_mail's ``window``): at most that many draws beyond
        the completed ones are in flight, so the first batches complete first.  "auto": 128 with the doubling plan (small
        batches, all gather CTAs resident at once), 400 with one wave per batch (a shallower HBM queue: the K4 launches
        that run under the gather keep pace with its waves); 0: no limit.
        k4_priority: K4 and K2b run on a high-priority stream of the loop (the gather's CTAs queue for every free slot of
        every SM; without priority the target kernels' CTAs wait behind them), joined back into the caller's stream.
        waves_when_eager: the waves are a schedule for the CAPTURED step (one graph replay per step).  Issued eagerly a
        step is bound by the host's launch path (~25 ctypes calls at batch 32), and the waves' extra launches, events and
        stream switches cost more there than the overlap returns (2.7 against 4.6 M transitions/s), so outside a capture
        ``step()`` issues the single gather launch unless this is set (the tests set it).
        pdl_at_joins: the K4 that waits for a wave keeps its programmatic-launch attribute (it executes griddepcontrol.wait
        before it reads anything, so every predecessor is complete whichever way the edge is typed): 67.2 against 68.2 us
        per batch-32 step.  False: those K4 launches are plain stream-ordered launches.
        replacement=False: every batch holds B distinct records, drawn by a0_pt_sample_unique (the law of the
        reference's torch.multinomial(priority[:top], B, replacement=False), replay.py:41-43) from the sampler's own
        Philox stream (``rng_seed``; drawn from torch's default generator when None), and gathered by one plain K3
        launch: the overlapped and waved schedules (``overlap_sample_gather``, default on only with replacement)
        are for the stratified draw."""
        assert algo in ALGOS, algo
        self.lib = _lib.load()
        self.rp, self.algo, self.B, self.L, self.A = replay, algo, int(batch_size), int(learner_steps), int(action_dim)
        self.total = T = self.L * self.B
        self.dev = dev = replay.device
        self.variant = int(variant)
        self.replacement = bool(replacement)
        if not self.replacement:
            if overlap_sample_gather:
                raise ValueError("ReplayTargetLoop(replacement=False) gathers with one plain launch: the overlapped / waved "
                                 "sample-gather schedules draw with replacement only")
            if self.B > 1024:
                raise ValueError(f"ReplayTargetLoop(replacement=False) takes batches of at most 1024 records, not {self.B}")
            if rng_seed is None:
                rng_seed = int(torch.randint(-2 ** 63, 2 ** 63 - 1, (1,), dtype=torch.int64).item())
        elif overlap_sample_gather is None:
            overlap_sample_gather = True
        self.overlap_sg = bool(overlap_sample_gather) and int(variant) == 0
        self.early_update = bool(early_update)      # step(): K2b starts under the last K4 (a0_pt_update_overlapped)
        self.rng_seed = None if rng_seed is None else int(rng_seed) & 0xFFFFFFFFFFFFFFFF
        self.n = int(n_step if n_step is not None else replay.n_gather)
        self.gamma = float(discount if discount is not None else replay.gamma)
        self.gamma_n = float(np.float32(self.gamma ** self.n))
        self.per = replay.prioritize if per is None else bool(per)
        self.double_q = bool(double_q)
        self.alpha, self.eps = float(alpha), float(eps)
        self.c51, self.mdqn = c51, mdqn
        e = lambda *s, dt=torch.float32: torch.empty(*s, dtype=dt, device=dev)
        self.u = e(T)
        self.idx = e(T, dt=torch.int64); self.prio = e(T); self.w = e(T)
        self.frames = frames if frames is not None else e(T, 8 * replay.F, dt=torch.uint8)
        self.act = e(T, dt=torch.int64); self.r64 = e(T, dt=torch.float64); self.r32 = e(T)
        self.d8 = e(T, dt=torch.uint8); self.d32 = e(T); self.boot = e(T, dt=torch.int64)
        self.loss = e(T); self.newp = e(T) if want_prio else None
        self.o = outputs
        self.grad = torch.empty_like(self.o["online"])
        self.frac = e(T) if algo == "fqf" else None
        self.gtau = e(T, self.o["taus"].shape[1]) if algo == "fqf" else None
        self.waves = self._wave_plan(gather_waves) if self.overlap_sg else None
        self.pdl_at_joins = bool(pdl_at_joins)
        self.waves_when_eager = bool(waves_when_eager)
        if self.waves:
            self.side = torch.cuda.Stream(device=dev)
            self.fast = torch.cuda.Stream(device=dev, priority=-1) if k4_priority else None
            self.wave_ev = [torch.cuda.Event() for _ in self.waves]
            self._join = {b0: j for j, (b0, _, _, _) in enumerate(self.waves)}      # first batch of wave j -> j
            per_batch = self.B * 16 * replay.F >= 10_000_000     # wave_plan's criterion: a batch's gather outlasts a K4
            # measured on B200 (profiles/r02s3_gather_waves_ab.json): 128 draws in flight feed a batch-32 K4 chain in order
            # at 67.9 us per step (96: 71.4, no limit: 71.0); 400 of the ~1036 resident gather CTAs in flight keep the
            # batch-512 step's K4 launches on pace with the waves at 216 us (no limit: 238, 320: 233, 480: 223)
            self.window = (400 if per_batch else 128) if gather_window == "auto" else int(gather_window or 0)
        n_gather = len(self.waves) if self.waves else 1
        # the waved step writes its priorities back in two halves when the count fits one CTA: a0_pt_update_plan on the side
        # stream after the last wave, and a0_pt_update_apply under the last K4 (a0_pt_update_overlapped's chunk
        # schedule otherwise).  The plan starts when the last wave is complete; the K4 that waits for it comes at least one
        # link after the one that waits for that wave, and 4 links before the end.  (launches_per_step leaves the plan out.)
        self._plan_join = max(self.waves[-1][0] + 1, self.L - 4) if self.waves else self.L
        self._use_plan = self._use_plan_default = self.per and self.early_update and T <= _lib.K2B_PLAN_MAX and self._plan_join < self.L
        if self._use_plan:
            self.plan = torch.empty(_lib.K2B_PLAN_BYTES, dtype=torch.uint8, device=dev)
            self.plan_ev = torch.cuda.Event()
        self.launches_per_step = 1 + n_gather + self.L + (1 if self.per else 0)     # our kernels (uniform_ is torch's)
        self._k4 = self._k4_early = None
        self._k4_all = None
        self.graph = None
        self.report = []          # pinned host (indices, losses) pairs filled by K2b: bind_report()
        self._report_dev = []
        self.graphs = []          # one captured step per report slot

    # ------------------------------------------------------------------ single launches
    def _st(self):
        return _lib.stream_ptr(self.dev)      # evaluated at call time: the capture stream inside a graph

    def sample(self):
        """K2a: L stratified batches + IS weights (top/beta from the device: push_dynamic first)."""
        rp = self.rp
        if not self.replacement:
            _lib.check(self.lib.a0_pt_sample_unique(rp.h, self.rng_seed, -1, self.total, self.B, -1.0, float(rp.beta), 0.0,
                                                    0 if self.per else 1, self.idx.data_ptr(), self.prio.data_ptr(),
                                                    self.w.data_ptr(), None, self._st()), "a0_pt_sample_unique")
            return
        if self.rng_seed is not None:
            _lib.check(self.lib.a0_pt_sample_rng(rp.h, self.rng_seed, -1, self.total, self.B, -1.0, float(rp.beta), 0.0,
                                                 0 if self.per else 1, self.idx.data_ptr(), self.prio.data_ptr(),
                                                 self.w.data_ptr(), None, self._st()), "a0_pt_sample_rng")
            return
        _lib.check(self.lib.a0_pt_sample(rp.h, self.u.data_ptr(), self.total, self.B, -1.0, float(rp.beta), 0.0,
                                         0 if self.per else 1, self.idx.data_ptr(), self.prio.data_ptr(),
                                         self.w.data_ptr(), self._st()), "a0_pt_sample")

    def gather(self, idx_ptr=None, out_ptr=None, count=None, variant=None):
        """K3: the sampled transitions' stacks + n-step scalars into the static buffers."""
        _lib.check(self.lib.a0_rb_gather(self.rp.h, idx_ptr or self.idx.data_ptr(), count or self.total, self.n, self.gamma,
                                         out_ptr or self.frames.data_ptr(), self.act.data_ptr(), self.r64.data_ptr(),
                                         self.r32.data_ptr(), self.d8.data_ptr(), self.d32.data_ptr(), self.boot.data_ptr(),
                                         self.variant if variant is None else variant, self._st()), "a0_rb_gather")

    def sample_gather(self):
        """K2a + K3 overlapped (a0_rb_sample_gather): same outputs as sample() followed by gather()."""
        rp = self.rp
        _lib.check(self.lib.a0_rb_sample_gather(
            rp.h, None if self.rng_seed is not None else self.u.data_ptr(), self.rng_seed or 0, -1, self.total, self.B, -1.0,
            float(rp.beta), 0.0, 0 if self.per else 1, self.idx.data_ptr(), self.prio.data_ptr(), self.w.data_ptr(), self.n,
            self.gamma, self.frames.data_ptr(), self.act.data_ptr(), self.r64.data_ptr(), self.r32.data_ptr(),
            self.d8.data_ptr(), self.d32.data_ptr(), self.boot.data_ptr(), self._st()), "a0_rb_sample_gather")

    def _wave_plan(self, spec):
        return wave_plan(self.L, self.B, self.rp.F, spec)

    def sample_gather_waves(self, plan=False):
        """K2a + the gather in waves on the side stream (a0_rb_sample_mail, a0_rb_gather_mail per wave, an event after
        each): same outputs as sample_gather().  The caller's stream joins wave by wave (``_wait_wave``).  plan: then the
        first half of the write-back (a0_pt_update_plan) on the same stream, and ``plan_ev`` after it."""
        rp, lib = self.rp, self.lib
        main = torch.cuda.current_stream(self.dev)
        self.side.wait_stream(main)           # everything before this step (the previous write-back, the ingest)
        with torch.cuda.stream(self.side):
            st = self._st()
            _lib.check(lib.a0_rb_sample_mail(rp.h, None if self.rng_seed is not None else self.u.data_ptr(), self.rng_seed or 0, -1,
                                             self.total, self.B, -1.0, float(rp.beta), 0.0, 0 if self.per else 1, self.idx.data_ptr(),
                                             self.prio.data_ptr(), self.w.data_ptr(), st), "a0_rb_sample_mail")
            for j, (_, _, lo, cnt) in enumerate(self.waves):
                _lib.check(lib.a0_rb_gather_mail(rp.h, lo, cnt, self.window, self.n, self.gamma, self.frames.data_ptr(), self.act.data_ptr(),
                                                 self.r64.data_ptr(), self.r32.data_ptr(), self.d8.data_ptr(), self.d32.data_ptr(),
                                                 self.boot.data_ptr(), st), "a0_rb_gather_mail")
                self.wave_ev[j].record(self.side)
            if plan:
                _lib.check(lib.a0_pt_update_plan(rp.h, self.idx.data_ptr(), self.total, self.plan.data_ptr(), st), "a0_pt_update_plan")
                self.plan_ev.record(self.side)

    def _wait_wave(self, j):
        torch.cuda.current_stream(self.dev).wait_event(self.wave_ev[j])

    def _common(self, lo, count):
        s = slice(lo, lo + count)
        p = lambda t: t[s].data_ptr()
        return _lib.LossCommon(B=count, A=self.A, action=p(self.act), reward=p(self.r32), done=p(self.d32), weight=p(self.w),
                               gamma_n=self.gamma_n, alpha=self.alpha, eps=self.eps, loss=p(self.loss), prio=p(self.newp) if self.newp is not None else None,
                               # uniform replay keeps no running max loss: a K4 that raised max_p would make later
                               # appends heavier than earlier ones (leaf = max_p^alpha) and the draw non-uniform
                               max_p=self.rp.max_p_tensor.data_ptr() if self.per else None), s

    def _bind(self, lo, count, early=False):
        """(function, argument tuple) of the K4 launch over rows [lo, lo+count): the a0_loss_common_t block
        and the sliced device pointers are built once, so a launch is a single ctypes call.  early: a link of
        ``early_links`` (C51 only)."""
        lib, o, algo = self.lib, self.o, self.algo
        c, s = self._common(lo, count)
        p = lambda t: t[s].data_ptr()
        qsel = p(o["qsel"]) if (self.double_q or algo in ("iqn", "fqf")) and algo != "mdqn" else None
        if algo == "dqn":
            a = (lib.a0_loss_dqn, (C.byref(c), p(o["online"]), p(o["tgt_next"]), qsel, p(self.grad)))
        elif algo == "mdqn":
            a = (lib.a0_loss_mdqn, (C.byref(c), p(o["online"]), p(o["tgt_next"]), p(o["tgt_cur"]), self.mdqn[0], self.mdqn[1],
                                    p(self.grad)))
        elif algo == "c51":
            M, vmin, vmax = self.c51
            if early:
                a = (lib.a0_loss_c51_linked, (C.byref(c), p(o["online"]), p(o["tgt_next"]), qsel, o["atoms"].data_ptr(), M, vmin,
                                              vmax, p(self.grad), None, _lib.C51_EARLY))
            else:
                a = (lib.a0_loss_c51, (C.byref(c), p(o["online"]), p(o["tgt_next"]), qsel, o["atoms"].data_ptr(), M, vmin, vmax,
                                       p(self.grad), None))
        elif algo == "qr":
            N = o["online"].shape[2]
            a = (lib.a0_loss_quantile, (C.byref(c), 0, p(o["online"]), p(o["tgt_next"]), None, qsel, o["tgt_next"].shape[2], N,
                                        p(self.grad), None, None, None, None))
        elif algo == "iqn":
            a = (lib.a0_loss_quantile, (C.byref(c), 1, p(o["online"]), p(o["tgt_next"]), p(o["taus"]), qsel,
                                        o["tgt_next"].shape[1], o["online"].shape[1], p(self.grad), None, None, None, None))
        else:
            F_ = o["online"].shape[1]
            a = (lib.a0_loss_quantile, (C.byref(c), 1, p(o["online"]), p(o["tgt_next"]), p(o["taus_hat"]), qsel, F_, F_,
                                        p(self.grad), p(o["q_bar"]), p(o["taus"]), p(self.frac), p(self.gtau)))
        return c, a

    def target_loss(self, k, early=False):
        """K4 for batch k: per-sample loss, gradient w.r.t. the online output, new priorities.  early: batch k's link is
        one of ``early_links`` (its inputs but the network outputs are read before its wait; C51's short-chain kernel)."""
        if self._k4 is None:
            self._k4 = [self._bind(k_ * self.B, self.B) for k_ in range(self.L)]
            self._k4_early = [self._bind(k_ * self.B, self.B, early=True) for k_ in range(self.L)] if self.algo == "c51" else None
        fn, args = (self._k4_early if early and self._k4_early else self._k4)[k][1]
        rc = fn(*args, self._st())
        if rc:
            _lib.check(rc, "a0_loss_" + self.algo)

    def target_loss_all(self):
        """All L batches in ONE K4 launch.  Valid only when every batch's network outputs exist before
        the first update, which a training loop cannot offer (evaluation, or measuring how much of a
        batch-32 step is launch latency)."""
        if self._k4_all is None:
            self._k4_all = self._bind(0, self.total)
        fn, args = self._k4_all[1]
        rc = fn(*args, self._st())
        if rc:
            _lib.check(rc, "a0_loss_" + self.algo)

    def bind_report(self, slots=2):
        """Page-locked host buffers for the step's result -- what ``BaseLearner.train`` returns on the
        CPU (agent.py:163-169: per-sample losses and indices).  With a report slot, K2b stores them
        straight into host memory (a0_pt_update_report) instead of two device-to-host copies being
        queued behind the step; ``slots`` buffers let the host read step s-1 while step s runs.
        Returns the list of (indices i64[L*B], losses f32[L*B]) pinned CPU tensor pairs."""
        self.report = [(torch.empty(self.total, dtype=torch.int64).pin_memory(),
                        torch.empty(self.total, dtype=torch.float32).pin_memory()) for _ in range(int(slots))]
        self._report_dev = [(_lib.host_map(i), _lib.host_map(l)) for i, l in self.report]
        return self.report

    def update(self, slot=None, after_k4=False):
        """K2b: priority[idx] = (loss+eps)^alpha for all L batches, max_p (replay.py:55-59).  ``slot``:
        also hand indices and losses to the host through report buffer ``slot`` (bind_report)."""
        if self.per and self.early_update and after_k4:
            # the launch before this one is the step's last K4 and the indices were written by the draw, several
            # launches earlier: K2b may start under that K4 (a0_pt_update_overlapped)
            ri, rl = self._report_dev[slot] if slot is not None else (None, None)
            _lib.check(self.lib.a0_pt_update_overlapped(self.rp.h, self.idx.data_ptr(), self.loss.data_ptr(), self.total, self.alpha,
                                                        self.eps, ri, rl, self._st()), "a0_pt_update_overlapped")
            return
        if self.per and slot is not None:
            ri, rl = self._report_dev[slot]
            _lib.check(self.lib.a0_pt_update_report(self.rp.h, self.idx.data_ptr(), self.loss.data_ptr(), self.total, self.alpha,
                                                    self.eps, ri, rl, self._st()), "a0_pt_update_report")
            return
        if self.per:
            _lib.check(self.lib.a0_pt_update(self.rp.h, self.idx.data_ptr(), self.loss.data_ptr(), self.total, self.alpha,
                                             self.eps, self._st()), "a0_pt_update")
        if slot is not None:          # uniform replay has no K2b launch to carry the report
            self.report[slot][0].copy_(self.idx, non_blocking=True)
            self.report[slot][1].copy_(self.loss, non_blocking=True)

    def _apply(self, slot=None):
        """Second half of the planned write-back (a0_pt_update_apply), launched right after the step's last K4."""
        ri, rl = self._report_dev[slot] if slot is not None else (None, None)
        _lib.check(self.lib.a0_pt_update_apply(self.rp.h, self.idx.data_ptr(), self.loss.data_ptr(), self.total, self.alpha,
                                               self.eps, self.plan.data_ptr(), ri, rl, self._st()), "a0_pt_update_apply")

    # ------------------------------------------------------------------ whole steps
    def _targets_and_update(self, fused_k4, slot, update=True, planned=False):
        """The K4 launches of a step whose gather runs in waves (each waits for the wave that holds its batch), then K2b.
        planned: the K4 ``_plan_join`` also waits for the plan (it executes griddepcontrol.wait before anything else, so the
        plan is complete when the apply, launched under the last K4, starts), and the apply is the write-back."""
        if fused_k4:
            for j in range(len(self.waves)):
                self._wait_wave(j)
            self.target_loss_all()
            if update:
                self.update(slot, after_k4=True)
            return
        early = early_links(self.L, self.waves, self._plan_join if planned else None)
        for k in range(self.L):
            j = self._join.get(k)
            join_plan = planned and k == self._plan_join
            if join_plan:
                torch.cuda.current_stream(self.dev).wait_event(self.plan_ev)
            if (j is None and not join_plan) or self.pdl_at_joins:
                if j is not None:
                    self._wait_wave(j)
                self.target_loss(k, early=k in early)
            else:
                # the K4 that joins wave j (or the plan) has more than one predecessor: launched without the
                # programmatic attribute unless pdl_at_joins
                if j is not None:
                    self._wait_wave(j)
                mask = C.c_int64(0)
                _lib.check(self.lib.a0_get_option(_lib.OPT_PDL, C.byref(mask)), "a0_get_option")
                self.lib.a0_set_option(_lib.OPT_PDL, mask.value & ~1)
                try:
                    self.target_loss(k)
                finally:
                    self.lib.a0_set_option(_lib.OPT_PDL, mask.value)
        if planned:
            self._apply(slot)
        elif update:
            self.update(slot, after_k4=True)

    def step(self, fused_k4=False, slot=None, update=True):
        """update=False: everything but the priority write-back (StaleByOneLoop issues it during the next step)."""
        if self.rng_seed is None:
            self.u.uniform_()
        if self.waves and (self.waves_when_eager or torch.cuda.is_current_stream_capturing()):
            planned = update and self._use_plan and not fused_k4
            self.sample_gather_waves(plan=planned)
            if self.fast is None:
                self._targets_and_update(fused_k4, slot, update, planned)
                return
            main = torch.cuda.current_stream(self.dev)
            self.fast.wait_stream(main)           # the network outputs, the previous step
            with torch.cuda.stream(self.fast):
                self._targets_and_update(fused_k4, slot, update, planned)
            main.wait_stream(self.fast)
            return
        if self.overlap_sg:
            self.sample_gather()
        else:
            self.sample()
            self.gather()
        if fused_k4:
            self.target_loss_all()
        else:
            for k in range(self.L):
                self.target_loss(k)
        if update:
            self.update(slot, after_k4=True)

    def capture(self, warm=3, fused_k4=False):
        """Warm up, then capture one step into a CUDA graph (returned; also kept as ``self.graph``)."""
        self.rp.push_dynamic()
        for _ in range(warm):
            self.step(fused_k4)
        torch.cuda.synchronize(self.dev)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self.step(fused_k4)
        self.graph = g
        return g

    def capture_reporting(self, warm=3):
        """One captured step per report slot (bind_report first): ``run(slot=s)`` replays the graph whose
        K2b writes the result into host buffer ``s``."""
        assert self.report, "bind_report() first"
        self.rp.push_dynamic()
        for _ in range(warm):
            self.step(slot=0)
        torch.cuda.synchronize(self.dev)
        self.graphs = []
        for s in range(len(self.report)):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self.step(slot=s)
            self.graphs.append(g)
        return self.graphs

    def run(self, slot=None, publish=True):
        """One step: publishes top/beta (``publish=False`` when the ingest already did:
        ``append_steps(publish_dynamic=True)``), then replays the captured graph (or issues the
        launches).  ``slot``: the report buffer this step's result goes to."""
        if publish:
            self.rp.push_dynamic()
        if slot is not None and self.graphs:
            self.graphs[slot].replay()
        elif slot is None and self.graph is not None:
            self.graph.replay()
        else:
            self.step(slot=slot)


class StaleByOneLoop:
    """Opt-in schedule of the same inner loop with the priority write-back of step s taken off the critical
    path: K2b(s) runs on a side stream WHILE step s+1 draws and gathers (K2a + K3), so step s+1 samples with
    priorities that are one step stale.  The reference itself samples with stale priorities -- its 2 DataLoader
    workers and 3-deep prefetch queue draw several batches ahead of the updates (trainer.py:64-70,83-87; SURVEY
    Q4) -- so this is inside its semantics, but it is NOT the default: ``ReplayTargetLoop`` applies every update
    before the next draw and is what the parity tests and bench.py's ``value`` use.

    Two ``ReplayTargetLoop`` buffer sets alternate (step s writes set s % 2); graph p replays
        main stream:  K2a + K3 into set p  ->  K4 x L on set p
        side stream:  K2b on set 1-p (the previous step's indices and losses)
    and joins both.  Updates are applied in step order (each K2b waits for its predecessor through the graph
    replays), duplicates keep last-writer-wins, the tree stays node == fl32(left + right) at every replay
    boundary.  A draw that races with a write-back can see a parent that is newer or older than its children:
    every decision of the descent still moves to a child whose mass was positive when it was read, and K2b never
    zeroes a leaf, so every drawn index is a live record (tested).

    Call ``flush()`` before ``ReplayDataset.save``: until then the last step's priority write-back is still pending
    and the checkpoint would miss it."""

    def __init__(self, replay, algo, batch_size, learner_steps, action_dim, outputs, **kw):
        kw = dict(kw)
        kw.setdefault("rng_seed", 1)
        self.loops = [ReplayTargetLoop(replay, algo, batch_size, learner_steps, action_dim, outputs, **kw) for _ in range(2)]
        self.rp = replay
        self.total = self.loops[0].total
        self.side = torch.cuda.Stream(device=replay.device)
        self.graphs = None
        self.s = 0
        self.launches_per_step = self.loops[0].launches_per_step

    def _step(self, p, first=False):
        cur, prev = self.loops[p], self.loops[1 - p]
        main = torch.cuda.current_stream(self.rp.device)
        if not first:
            self.side.wait_stream(main)
            with torch.cuda.stream(self.side):
                prev.update()
        cur.step(update=False)               # K2a + gather (in waves) + K4 x L into set p
        if not first:
            main.wait_stream(self.side)

    def capture(self, warm=2):
        self.rp.push_dynamic()
        self._step(0, first=True)
        for i in range(warm):
            self._step((i + 1) % 2)
        torch.cuda.synchronize(self.rp.device)
        self.s = warm + 1
        self.graphs = {}
        for q in range(2):                              # the graph that writes buffer set q (steps with s % 2 == q)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._step(q)
            self.graphs[q] = g
        return self.graphs

    def run(self, publish=True):
        """One step (replays the graph of the current parity); the step's own write-back happens during the next."""
        if publish:
            self.rp.push_dynamic()
        if self.graphs is None:
            self._step(self.s % 2, first=self.s == 0)
        else:
            self.graphs[self.s % 2].replay()
        self.s += 1

    def current(self):
        """The buffer set the LAST run() wrote (indices, losses, gradients ...)."""
        return self.loops[(self.s - 1) % 2]

    def flush(self):
        """Apply the write-back of the last step (nothing is pending afterwards)."""
        self.current().update()
