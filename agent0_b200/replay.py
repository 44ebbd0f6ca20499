"""HBM-resident replay shard behind the reference's ``ReplayDataset`` interface.

Drop-in surface (agent0/deepq/replay.py:14-59): ``ReplayDataset(cfg)``, ``extend(transitions)``,
``__len__``, ``top``, ``beta``, ``max_p``, ``priority`` (an object with ``.sum()``),
``update_priority(ids, priorities)``.  New: ``sample(batch_size, k_batches)`` replaces the
DataLoaderX/DataPrefetcher pump (agent0/deepq/trainer.py:63-72, agent0/common/utils.py:31-61) and
returns device-resident tensors in the reference's 6-tuple order plus the fused IS weights;
``append_steps`` is the native single-frame ingest for actors that feed the shard directly.

Everything on the data path is native code from libagent0_b200.so: the CUDA kernels (K1 append,
K2a sample, K2b update, K3 gather) and the C++ ring index + pinned staging behind
``a0_rb_ingest_steps`` / ``a0_rb_ingest_plan``; this module marshals arguments.  There is no CPU
fallback.
"""
from __future__ import annotations

import ctypes as C
import json
import os
from collections import namedtuple

import numpy as np
import torch

from . import _lib
from .ring_index import NativeRingIndex, stack_delta, stream_map_arrays

Batch = namedtuple("Batch", ["frames", "actions", "rewards", "terminals", "priorities", "indices",
                             "weights", "rewards_f32", "terminals_f32", "boot_indices", "obs", "next_obs"],
                   defaults=(None, None))
Batch.__doc__ = """One or more sampled batches, device resident.  Fields 0..5 are the reference's
collated 6-tuple (frames u8[B,8*F], a i64, r f64, d bool, priority f32, idx i64; SURVEY 8b);
``weights`` are the IS weights of trainer.py:91-96, ``*_f32`` the .float() casts of trainer.py:88-90.
With ``normalized=`` sampling, ``frames`` is None and ``obs`` / ``next_obs`` are the learner's
f32 [B,4,H,W] inputs (agent.py:129-135: /255 and split, fused into the gather)."""
NORM_DIV, NORM_RECIP, NORM_NONE = 0, 1, 2      # a0_rb_gather_f32 norm_mode



def split_batches(batch, batch_size):
    """Per-update views of a multi-batch draw: a list of ``Batch`` tuples, one per learner update
    (torch.split makes all views of a field in one call)."""
    cols = [f.split(batch_size) if f is not None else None for f in batch]
    k = len(next(c for c in cols if c is not None))
    return [Batch(*[(c[i] if c is not None else None) for c in cols]) for i in range(k)]


def _is_prioritized(cfg):
    pol = cfg.replay.policy
    return getattr(pol, "name", str(pol)) == "prioritize"


class _LinearSchedule:
    """beta annealing with the semantics of agent0/common/utils.py:12-28: a call returns the
    current value and then advances by inc*steps, clamped at ``end``."""

    def __init__(self, start, end, steps):
        self.inc = (end - start) / float(steps)
        self.current, self.end = start, end
        self.bound = min if end > start else max

    def __call__(self, steps=1):
        val = self.current
        self.current = self.bound(self.current + self.inc * steps, self.end)
        return val


class _PrioritySum:
    """Stands in for the reference's ``replay.priority`` tensor where Trainer.step only calls
    ``.sum()`` on it (trainer.py:92): the sum is the tree root, already on the device."""

    def __init__(self, owner):
        self._o = owner

    def sum(self):
        return self._o.priority_sum()

    def leaves(self):
        return self._o.tree[self._o.P:self._o.P + self._o.size]


class ReplayDataset:
    def __init__(self, cfg, device=None, frame_capacity=None, native_nstep=False, compat_sum=False,
                 gather_variant=0, age_limit=None):
        """cfg: the reference's ExpConfig (or agent0_b200.config.ExpConfig; same attribute names).

        native_nstep=False: ``extend`` receives the reference actor's already n-step-folded
        entries, so records are gathered with a 1-step window.  native_nstep=True: ``append_steps``
        receives raw 1-step transitions and K3 folds ``cfg.learner.n_step_q`` steps.
        compat_sum=True reproduces the reference's IS-weight denominator over never-written slots
        (SURVEY Q3); the default uses the sum over live priorities.
        """
        self.cfg = cfg
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise RuntimeError("agent0_b200.ReplayDataset needs a CUDA device (no CPU fallback)")
        if device is None:
            dv = getattr(cfg.device, "value", cfg.device)
            device = torch.device(dv if str(dv).startswith("cuda") else "cuda")
        self.device = torch.device(device)
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.size = int(cfg.replay.size)
        obs_shape = tuple(cfg.obs_shape)
        self.stack = int(obs_shape[0])
        assert self.stack == 4, "the kernels are specialised for 4-frame stacks (FrameStack(4))"
        self.frame_shape = obs_shape[1:]
        self.F = int(np.prod(self.frame_shape))
        assert self.F % 16 == 0, "frame bytes must be a multiple of 16"
        self.n_gather = int(cfg.learner.n_step_q) if native_nstep else 1
        self.gamma = float(cfg.learner.discount)
        if frame_capacity is None:
            frame_capacity = int(self.size * 1.0625) + 65536 if self.size >= 65536 else 4 * self.size + 64
        self.index = NativeRingIndex(self.size, frame_capacity, self.n_gather, age_limit)
        self.prioritize = _is_prioritized(cfg)
        # uniform replay: alpha = 0 makes every new leaf max_p^0 = 1 whatever max_p is (the reference's uniform
        # policy never reads priorities, trainer.py:95-96), so the tree descent draws records uniformly
        self.alpha = float(cfg.replay.alpha) if self.prioritize else 0.0
        self.eps = float(cfg.replay.eps)
        self.compat_sum = bool(compat_sum)
        self.gather_variant = int(gather_variant)
        if self.prioritize:
            self.beta_schedule = _LinearSchedule(cfg.replay.beta0, 1.0, cfg.trainer.total_steps)
            self.beta = cfg.replay.beta0
        else:
            self.beta = 1.0
        self.num_envs = int(cfg.actor.num_envs)

        h = C.c_void_p()
        _lib.check(self.lib.a0_rb_create(C.byref(h), self.size, frame_capacity, self.F, self.device.index),
                   "a0_rb_create")
        self.h = h
        self.P = int(self.lib.a0_rb_tree_leaves(h))
        dev = self.device
        # views of handle-owned memory keep the handle alive (owner=): a tensor handed to a learner or cached in
        # a captured graph must never outlive the allocation it points into
        self._owner = _lib.HandleOwner(self.lib, h)
        self.frames = _lib.device_view(self.lib.a0_rb_ptr(h, _lib.PTR_FRAMES), (frame_capacity, self.F), "|u1", dev, self._owner)
        self.tree = _lib.device_view(self.lib.a0_rb_ptr(h, _lib.PTR_TREE), (2 * self.P,), "<f4", dev, self._owner)
        self.max_p_tensor = _lib.device_view(self.lib.a0_rb_ptr(h, _lib.PTR_MAX_P), (1,), "<f4", dev, self._owner)
        self.priority = _PrioritySum(self)
        ex = C.c_void_p()
        _lib.check(self.lib.a0_ex_create(C.byref(ex), h, self.index.h), "a0_ex_create")
        self._ex = ex                                             # reference-tuple ingest (K6)

    # ------------------------------------------------------------------ reference surface
    def __len__(self):
        return self.index.top

    @property
    def top(self):
        return self.index.top

    @property
    def max_p(self):
        """Host copy of the running max loss (synchronises; the kernels use the device copy)."""
        return float(self.max_p_tensor.item())

    def priority_sum(self):
        root = self.tree[1]
        if self.compat_sum:
            return root + float(self.size - self.index.top)
        return root

    def __del__(self):
        try:
            if getattr(self, "_ex", None) is not None and self._ex.value:
                self.lib.a0_ex_destroy(self._ex)
                self._ex = None
            self.h = None          # a0_rb_destroy runs when the last view of the shard's memory is gone (HandleOwner)
            self._owner = None
        except Exception:
            pass

    # ------------------------------------------------------------------ ingest: reference tuples
    def extend(self, transitions, streams=None):
        """Reference-compatible ingest (replay.py:45-53): a list of (frames, action, reward, done)
        with frames = the 8-frame blob concat(st, st_next) as the reference actor ships it -- a
        python-lz4 block (agent.py:78-81) -- or the same 8 frames uncompressed (bytes / ndarray).
        Entries arrive step-major, env-minor, so entry i belongs to stream i % num_envs unless
        ``streams`` says otherwise.  One C call (a0_ex_extend): the compressed bytes are copied to
        the device, decoded and de-duplicated there (K6: a frame already held for the stream's
        previous entry is not stored again; matches are byte-verified, so they are bit-exact),
        and the new frames are appended from the decoded scratch by K1."""
        m = len(transitions)
        if m == 0:
            return
        if self.n_gather != 1:
            raise RuntimeError("extend() takes the reference actor's already n-step-folded entries; this shard was built "
                               "with native_nstep=True and folds n_step_q records again at gather time -- feed it with "
                               "append_steps / ShardActor instead")
        if streams is None:
            streams = self._default_streams(m)
        else:
            streams = np.ascontiguousarray(streams, dtype=np.int64)
        assert len(streams) == m
        helper = _lib.pyingest()
        if helper is not None:
            # the tuples are unpacked by a C loop over the list (csrc/a0_pyingest.c); the blobs are copied once,
            # from where the actor left them into the page-locked staging block
            w = self._unpack_ws(m, helper)
            if helper.a0_py_unpack(transitions, m, w["ptrs"].ctypes.data, w["lens"].ctypes.data, w["action"].ctypes.data,
                                   w["reward"].ctypes.data, w["done"].ctypes.data, w["views"].ctypes.data) != m:
                raise RuntimeError("extend(): could not unpack the transitions")      # (a Python exception is normally set)
            try:
                with torch.cuda.device(self.device):
                    _lib.check(self.lib.a0_ex_extend_v(self._ex, w["ptrs"].ctypes.data, w["lens"].ctypes.data, streams.ctypes.data,
                                                       w["action"].ctypes.data, w["reward"].ctypes.data, w["done"].ctypes.data, m,
                                                       self.alpha, _lib.stream_ptr(self.device)), "a0_ex_extend")
            finally:
                helper.a0_py_release(m, w["views"].ctypes.data)
        else:
            blobs, action, reward, done = zip(*transitions)
            if not all(type(b) is bytes for b in blobs):
                blobs = [b if isinstance(b, (bytes, bytearray)) else np.ascontiguousarray(b, dtype=np.uint8).tobytes() for b in blobs]
            lens = np.fromiter(map(len, blobs), dtype=np.int64, count=m)
            joined = b"".join(blobs)
            action = np.asarray(action, dtype=np.int64)
            reward = np.asarray(reward, dtype=np.float64)
            done = np.asarray(done, dtype=np.bool_)
            with torch.cuda.device(self.device):
                _lib.check(self.lib.a0_ex_extend(self._ex, joined, lens.ctypes.data, streams.ctypes.data, action.ctypes.data,
                                                 reward.ctypes.data, done.ctypes.data, m, self.alpha,
                                                 _lib.stream_ptr(self.device)), "a0_ex_extend")
        if self.prioritize:
            self.beta = self.beta_schedule(m)

    def _default_streams(self, m):
        """entry i of an extend() call belongs to stream i % num_envs (the actor's order, agent.py:78)"""
        s = getattr(self, "_streams_cache", None)
        if s is None or len(s) < m:
            s = self._streams_cache = np.arange(max(m, 4096), dtype=np.int64) % self.num_envs
        return s[:m]

    def _unpack_ws(self, m, helper):
        w = getattr(self, "_unpack_cache", None)
        if w is None or len(w["lens"]) < m:
            cap = max(m, 2048)
            w = self._unpack_cache = dict(ptrs=np.zeros(cap, dtype=np.uint64), lens=np.zeros(cap, dtype=np.int64),
                                          action=np.zeros(cap, dtype=np.int64), reward=np.zeros(cap, dtype=np.float64),
                                          done=np.zeros(cap, dtype=np.uint8),
                                          views=np.zeros(cap * int(helper.a0_py_buffer_size()), dtype=np.uint8))
        return w

    def extend_timing(self):
        """Microseconds of the last ``extend``: host staging, wait for the device decode + label, host
        resolve + plan, append launches, device time of decode + label, entries."""
        out = np.zeros(6, dtype=np.float32)
        _lib.check(self.lib.a0_ex_last_timing(self._ex, out.ctypes.data), "a0_ex_last_timing")
        return dict(zip(("stage_us", "wait_us", "plan_us", "launch_us", "device_decode_label_us", "entries"), out.tolist()))

    def decode_entries(self, blobs):
        """K6a alone (tests, bench): python-lz4 blocks -> u8 [m, 8*F] on the device + i32 status per entry."""
        m = len(blobs)
        lens = np.fromiter(map(len, blobs), dtype=np.int64, count=m)
        out = torch.empty((m, 8 * self.F), dtype=torch.uint8, device=self.device)
        status = np.zeros(m, dtype=np.int32)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.a0_ex_decode(self._ex, b"".join(blobs), lens.ctypes.data, m, out.data_ptr(), status.ctypes.data,
                                             _lib.stream_ptr(self.device)), "a0_ex_decode")
        return out, status

    def _ingest_plan(self, plan, frames_ptr, new_src, flags):
        src = None
        if new_src is not None and len(new_src):
            new_src = np.ascontiguousarray(new_src, dtype=np.int64)
            src = new_src.ctypes.data
        with torch.cuda.device(self.device):
            _lib.check(self.lib.a0_rb_ingest_plan(self.h, C.byref(plan), frames_ptr, src, flags, self.alpha,
                                                  _lib.stream_ptr(self.device)), "a0_rb_ingest_plan")

    # ------------------------------------------------------------------ ingest: native 1-step
    def _frames_arg(self, frames, count, pinned_stable=False):
        """(keepalive, pointer, flags) of `count` frames given as a host array, a CPU tensor or a
        CUDA tensor."""
        if isinstance(frames, torch.Tensor):
            assert frames.dtype == torch.uint8 and frames.numel() == count * self.F
            t = frames if frames.is_contiguous() else frames.contiguous()
            if t.is_cuda:
                return t, t.data_ptr(), _lib.INGEST_FRAMES_ON_DEVICE
            return t, t.data_ptr(), (_lib.INGEST_FRAMES_PINNED if pinned_stable and t.is_pinned() else 0)
        a = np.ascontiguousarray(frames, dtype=np.uint8)
        assert a.size == count * self.F
        return a, a.ctypes.data, 0

    def reset_streams(self, streams, stacks):
        """Give streams their initial observation stack (u8 [k,4,H,W], host or device)."""
        streams = np.asarray(streams, dtype=np.int64)
        k = len(streams)
        ix = self.index
        seqs = ix.head_fs + np.arange(4 * k, dtype=np.int64)
        for i, sid in enumerate(streams):
            ix.set_stack(int(sid), seqs[4 * i:4 * i + 4])
        # frames only, no records
        z = np.zeros(0, dtype=np.int64)
        plan = ix.plan_native(z, np.zeros((0, 8), dtype=np.int64), 4 * k, z, z.astype(np.float64), z.astype(np.bool_))
        keep, ptr, flags = self._frames_arg(stacks, 4 * k)
        self._ingest_plan(plan, ptr, None, flags)

    def append_steps(self, streams, n_new, new_frames, action, reward, done, pinned_stable=False, copy_stream=False,
                     publish_dynamic=False):
        """Native ingest.  For each transition (in order) the observation is the stream's current
        stack and the next observation is that stack shifted by ``n_new`` (0..4) new frames taken,
        in order, from ``new_frames`` (u8 [sum(n_new), H, W]: host array, CPU tensor or CUDA
        tensor).  ``done`` follows the reference's rule (terminal | life_loss) & ~truncated
        (agent.py:57-62).  One C call: index update, staging, H2D copy, K2b marks and K1 append
        (one launch for a step-sized append).
        ``pinned_stable=True`` lets a page-locked CPU tensor be copied by DMA straight from the
        caller's buffer, which must then stay untouched until the current stream has passed.
        ``copy_stream=True`` issues the H2D DMA on the shard's own copy stream (the current stream
        waits for it), so it overlaps the kernels the current stream is still running.
        ``publish_dynamic=True``: the append launch also publishes top / beta / sum_offset for
        ``sample(dynamic=True)`` -- what a separate ``push_dynamic()`` launch would do."""
        streams = np.ascontiguousarray(streams, dtype=np.int64)
        n_new = np.ascontiguousarray(n_new, dtype=np.int64)
        action = np.ascontiguousarray(action, dtype=np.int64)
        reward = np.ascontiguousarray(reward, dtype=np.float64)
        done = np.ascontiguousarray(done, dtype=np.bool_)
        m = len(streams)
        keep, ptr, flags = self._frames_arg(new_frames, int(n_new.sum()), pinned_stable)
        if copy_stream and not (flags & _lib.INGEST_FRAMES_ON_DEVICE):
            flags |= _lib.INGEST_COPY_STREAM
        if self.prioritize:
            self.beta = self.beta_schedule(m)         # replay.py:53; the C call below does not read it
        with torch.cuda.device(self.device):
            if publish_dynamic:
                _lib.check(self.lib.a0_rb_ingest_steps_dyn(
                    self.h, self.index.h, streams.ctypes.data, n_new.ctypes.data, ptr, flags, action.ctypes.data,
                    reward.ctypes.data, done.ctypes.data, m, self.alpha, float(self.beta), 1 if self.compat_sum else 0,
                    _lib.stream_ptr(self.device)), "a0_rb_ingest_steps_dyn")
            else:
                _lib.check(self.lib.a0_rb_ingest_steps(
                    self.h, self.index.h, streams.ctypes.data, n_new.ctypes.data, ptr, flags, action.ctypes.data,
                    reward.ctypes.data, done.ctypes.data, m, self.alpha, _lib.stream_ptr(self.device)), "a0_rb_ingest_steps")

    def append_vector_step(self, obs, action, reward, done, obs_next, streams=None):
        """Convenience for a gymnasium-style vector step: derives ``n_new`` by comparing stacks."""
        E = obs.shape[0]
        streams = np.arange(E, dtype=np.int64) if streams is None else np.asarray(streams, dtype=np.int64)
        fresh = [i for i, s in enumerate(streams) if not self.index.has_stack(int(s))]
        if fresh:
            self.reset_streams(streams[fresh], obs[fresh])
        k = stack_delta(obs, obs_next)
        new = np.concatenate([obs_next[e, 4 - k[e]:] for e in range(E)]) if k.sum() else \
            np.zeros((0,) + tuple(obs.shape[2:]), dtype=np.uint8)
        self.append_steps(streams, k, new, action, reward, done)

    # ------------------------------------------------------------------ sample / gather
    def alloc_batch(self, total, normalized=None, obs_dtype=torch.float32):
        """Preallocated device buffers for ``total`` sampled transitions (``sample(..., out=)``):
        static addresses, as CUDA-graph capture of the consumer needs.  ``normalized`` (a NORM_*
        mode): obs / next_obs buffers of ``obs_dtype`` (float32 or bfloat16) instead of the u8 frames."""
        dev = self.device
        e = lambda dt, *s: torch.empty(s or (total,), dtype=dt, device=dev)
        shape = (total, self.stack) + tuple(self.frame_shape)
        assert obs_dtype in (torch.float32, torch.bfloat16)
        frames = e(torch.uint8, total, 8 * self.F) if normalized is None else None
        obs = e(obs_dtype, *shape) if normalized is not None else None
        nxt = e(obs_dtype, *shape) if normalized is not None else None
        return Batch(frames, e(torch.int64), e(torch.float64), e(torch.bool), e(torch.float32),
                     e(torch.int64), e(torch.float32), e(torch.float32), e(torch.float32), e(torch.int64), obs, nxt)

    def push_dynamic(self):
        """Publish top / beta / sum_offset to the device (stream-ordered) for ``sample(dynamic=True)``:
        a draw captured in a CUDA graph then follows the shard as it grows and beta anneals."""
        sum_offset = float(self.size - self.index.top) if self.compat_sum else 0.0
        with torch.cuda.device(self.device):
            _lib.check(self.lib.a0_rb_set_dynamic(self.h, float(self.index.top), float(self.beta), sum_offset,
                                                  _lib.stream_ptr(self.device)), "a0_rb_set_dynamic")

    def sample(self, batch_size=None, k_batches=1, u=None, indices=None, generator=None, out=None, dynamic=False,
               normalized=None, seed=None, call=-1, u_out=None, obs_dtype=None, replacement=True, stats_out=None):
        """Draw ``k_batches`` stratified batches (K2a) and gather them (K3).  ``u`` (f32 device
        tensor of k*B uniforms) or ``indices`` (i64, explicit record positions) make the draw
        reproducible for parity tests; otherwise uniforms come from torch's CUDA generator.
        ``out`` (from ``alloc_batch``) receives the result in place; ``dynamic=True`` reads top/beta
        from the device values last published by ``push_dynamic`` (for CUDA-graph capture).
        ``normalized`` (NORM_DIV / NORM_RECIP / NORM_NONE): gather straight into the learner's f32
        obs / next_obs inputs (K3 with the /255 + split of agent.py:129-135 fused in);
        ``obs_dtype=torch.bfloat16`` writes them as bf16(f32 value) for a mixed-precision CNN.
        ``seed`` (int): the sampler draws its own uniforms (Philox4x32-10 inside K2a, no separate RNG
        launch); ``call`` >= 0 names the call number, < 0 uses the shard's device-resident counter,
        which every launch -- or graph replay -- advances; ``u_out`` receives the uniforms.
        ``replacement=False``: no record twice in a batch, with the law of the reference's
        torch.multinomial(priority[:top], B, replacement=False) (replay.py:41-43; a0_pt_sample_unique, rows in draw
        order).  It takes its uniforms from the sampler's own Philox stream: without ``seed``, a 64-bit seed is drawn
        once from ``generator`` (or torch's default generator) and kept for the shard.  ``stats_out`` (i32 device
        tensor [k_batches, 2]) receives {rounds, candidates drawn} per batch."""
        B = int(batch_size or self.cfg.learner.batch_size)
        total = B * int(k_batches)
        dev = self.device
        if self.index.top <= 0:
            raise RuntimeError("sample() on an empty replay shard")
        if not replacement:
            if u is not None or indices is not None:
                raise ValueError("sample(replacement=False) draws its own uniforms: u= and indices= are not accepted")
            if B > 1024:
                raise ValueError(f"sample(replacement=False) takes batches of at most 1024 records, not {B}")
            if self.index.top < B:
                raise ValueError(f"sample(replacement=False): {B} distinct records asked of a shard that holds {self.index.top}")
            if stats_out is not None and stats_out.numel() < 2 * int(k_batches):
                raise ValueError("stats_out needs room for {rounds, candidates} of every batch")
            if seed is None:
                if getattr(self, "_unique_seed", None) is None:
                    gd = generator.device if generator is not None else "cpu"
                    self._unique_seed = int(torch.randint(-2 ** 63, 2 ** 63 - 1, (1,), dtype=torch.int64, device=gd,
                                                          generator=generator).item()) & 0xFFFFFFFFFFFFFFFF
                seed = self._unique_seed
        with torch.cuda.device(dev):
            stream = _lib.stream_ptr(dev)
            weights = out.weights if out is not None else torch.empty(total, dtype=torch.float32, device=dev)
            prio = out.priorities if out is not None else torch.empty(total, dtype=torch.float32, device=dev)
            if indices is None:
                idx = out.indices if out is not None else torch.empty(total, dtype=torch.int64, device=dev)
                sum_offset = float(self.size - self.index.top) if self.compat_sum else 0.0
                top = -1.0 if dynamic else float(self.index.top)
                if not replacement:
                    _lib.check(self.lib.a0_pt_sample_unique(
                        self.h, int(seed) & 0xFFFFFFFFFFFFFFFF, int(call), total, B, top, float(self.beta), sum_offset,
                        0 if self.prioritize else 1, _lib.ptr(idx), _lib.ptr(prio), _lib.ptr(weights),
                        _lib.ptr(stats_out, torch.int32), stream), "a0_pt_sample_unique")
                elif u is None and seed is not None:
                    _lib.check(self.lib.a0_pt_sample_rng(
                        self.h, int(seed) & 0xFFFFFFFFFFFFFFFF, int(call), total, B, top, float(self.beta), sum_offset,
                        0 if self.prioritize else 1, _lib.ptr(idx), _lib.ptr(prio), _lib.ptr(weights),
                        _lib.ptr(u_out, torch.float32), stream), "a0_pt_sample_rng")
                else:
                    if u is None:
                        u = torch.rand(total, dtype=torch.float32, device=dev, generator=generator)
                    _lib.check(self.lib.a0_pt_sample(
                        self.h, _lib.ptr(u, torch.float32), total, B, top, float(self.beta), sum_offset,
                        0 if self.prioritize else 1, _lib.ptr(idx), _lib.ptr(prio), _lib.ptr(weights), stream),
                        "a0_pt_sample")
            else:
                idx = indices.to(device=dev, dtype=torch.int64).contiguous()
                total = idx.numel()
                prio = self.tree[self.P + idx]
                weights = self.is_weights(prio, B) if self.prioritize else torch.ones_like(prio)
                if out is not None:
                    out.indices.copy_(idx); out.priorities.copy_(prio); out.weights.copy_(weights)
                    idx, prio, weights = out.indices, out.priorities, out.weights
            return self.gather(idx, prio, weights, out=out, normalized=normalized, obs_dtype=obs_dtype)

    def gather(self, idx, prio=None, weights=None, out=None, normalized=None, obs_dtype=None):
        dev = self.device
        total = idx.numel()
        if out is not None and out.obs is not None and normalized is None:
            normalized = NORM_DIV
        if obs_dtype is not None and normalized is None:
            normalized = NORM_DIV
        with torch.cuda.device(dev):
            if normalized is not None:
                return self._gather_f32(idx, prio, weights, out, int(normalized), obs_dtype)
            if out is not None:
                assert out.frames.shape[0] == total, "out= was allocated for a different number of transitions"
                frames, act, r64, d8, r32, d32, boot = (out.frames, out.actions, out.rewards, out.terminals, out.rewards_f32,
                                                        out.terminals_f32, out.boot_indices)
            else:
                frames = torch.empty((total, 8 * self.F), dtype=torch.uint8, device=dev)
                act = torch.empty(total, dtype=torch.int64, device=dev)
                r64 = torch.empty(total, dtype=torch.float64, device=dev)
                r32 = torch.empty(total, dtype=torch.float32, device=dev)
                d8 = torch.empty(total, dtype=torch.bool, device=dev)
                d32 = torch.empty(total, dtype=torch.float32, device=dev)
                boot = torch.empty(total, dtype=torch.int64, device=dev)
            _lib.check(self.lib.a0_rb_gather(
                self.h, _lib.ptr(idx, torch.int64), total, self.n_gather, self.gamma, frames.data_ptr(),
                act.data_ptr(), r64.data_ptr(), r32.data_ptr(), d8.data_ptr(), d32.data_ptr(), boot.data_ptr(),
                self.gather_variant, _lib.stream_ptr(dev)), "a0_rb_gather")
        return Batch(frames, act, r64, d8, prio, idx, weights, r32, d32, boot)

    def _gather_f32(self, idx, prio, weights, out, mode, obs_dtype=None):
        dev, total = self.device, idx.numel()
        shape = (total, self.stack) + tuple(self.frame_shape)
        if out is not None:
            assert out.obs is not None and out.obs.shape[0] == total, "out= was not allocated with normalized= for this size"
            assert obs_dtype is None or obs_dtype == out.obs.dtype, "out= was allocated with another obs_dtype"
            obs, nxt, act, r64, d8, r32, d32, boot = (out.obs, out.next_obs, out.actions, out.rewards, out.terminals,
                                                      out.rewards_f32, out.terminals_f32, out.boot_indices)
        else:
            e = lambda dt, *s: torch.empty(s or (total,), dtype=dt, device=dev)
            odt = obs_dtype or torch.float32
            assert odt in (torch.float32, torch.bfloat16)
            obs, nxt = e(odt, *shape), e(odt, *shape)
            act, r64, d8, r32 = e(torch.int64), e(torch.float64), e(torch.bool), e(torch.float32)
            d32, boot = e(torch.float32), e(torch.int64)
        bf16 = obs.dtype == torch.bfloat16
        fn = self.lib.a0_rb_gather_bf16 if bf16 else self.lib.a0_rb_gather_f32
        _lib.check(fn(
            self.h, _lib.ptr(idx, torch.int64), total, self.n_gather, self.gamma, obs.data_ptr(), nxt.data_ptr(), mode,
            act.data_ptr(), r64.data_ptr(), r32.data_ptr(), d8.data_ptr(), d32.data_ptr(), boot.data_ptr(),
            _lib.stream_ptr(dev)), "a0_rb_gather_bf16" if bf16 else "a0_rb_gather_f32")
        return Batch(None, act, r64, d8, prio, idx, weights, r32, d32, boot, obs, nxt)

    def global_is_weights(self, prio, batch, process_group):
        """IS weights of a draw re-normalised over the GLOBAL batch of all shards (dist.global_batch_is_weights:
        one all-reduce(MAX) of k_batches floats); the default weights of ``sample`` are normalised per shard."""
        from .dist import global_batch_is_weights
        return global_batch_is_weights(prio, self.tree[1], self.beta, batch, process_group)

    def is_weights(self, prio, batch):
        """trainer.py:91-94 with torch ops (used only when indices are given explicitly; the
        sampled path gets its weights from the K2a epilogue)."""
        w = (self.index.top * (prio / self.priority_sum())).pow(-self.beta).view(-1, batch)
        return (w / (w.max(dim=1, keepdim=True)[0] + 1e-8)).view(-1)

    # ------------------------------------------------------------------ priorities
    def update_priority(self, ids, priorities):
        """replay.py:55-59: priority[ids] = (loss+eps)^alpha; max_p = max(max_p, loss.max()).
        Device tensors stay on the device (no sync); host tensors are copied asynchronously."""
        if not self.prioritize or priorities is None:
            return
        dev = self.device
        ids = torch.as_tensor(ids).to(device=dev, dtype=torch.int64, non_blocking=True).contiguous()
        loss = torch.as_tensor(priorities).to(device=dev, dtype=torch.float32, non_blocking=True).contiguous()
        with torch.cuda.device(dev):
            _lib.check(self.lib.a0_pt_update(self.h, ids.data_ptr(), loss.data_ptr(), ids.numel(), self.alpha,
                                             self.eps, _lib.stream_ptr(dev)), "a0_pt_update")

    # ------------------------------------------------------------------ checkpoint
    def save(self, path):
        """Write the whole shard to ``path`` (a0_ckpt_save): frames of the resident window as K7 LZ4 blobs, records,
        priorities, max_p, the sampler's scalars and call counter, the ring index and the reference-tuple ingest's
        stream tails, plus beta, the beta schedule's position and the draw-without-replacement seed.  Synchronises
        the current stream; refused during a CUDA-graph capture.  A ``StaleByOneLoop`` must be ``flush()``ed first."""
        user = json.dumps(dict(beta=self.beta, beta_current=getattr(getattr(self, "beta_schedule", None), "current", None),
                               unique_seed=getattr(self, "_unique_seed", None))).encode()
        with torch.cuda.device(self.device):
            _lib.check(self.lib.a0_ckpt_save(self.h, self.index.h, self._ex, os.fsencode(os.fspath(path)), user, len(user),
                                             _lib.stream_ptr(self.device)), "a0_ckpt_save")

    def load(self, path):
        """Replace this shard's contents with a checkpoint written by ``save`` for a shard of the same config
        (a0_ckpt_load, into the buffers the shard already owns: CUDA graphs captured on it stay valid).  Raises
        RuntimeError on a mismatched or corrupt file; a file rejected before the frames are decoded leaves the shard
        as it was, a failure while they are decoded leaves it empty."""
        buf = C.create_string_buffer(1 << 16)
        n = C.c_int64(0)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.a0_ckpt_load(self.h, self.index.h, self._ex, os.fsencode(os.fspath(path)), buf, len(buf),
                                             C.byref(n), _lib.stream_ptr(self.device)), "a0_ckpt_load")
        self._apply_user(json.loads(buf.raw[:n.value].decode()) if n.value else {})

    def _apply_user(self, user):
        if "beta" in user:
            self.beta = user["beta"]
        if user.get("beta_current") is not None and getattr(self, "beta_schedule", None) is not None:
            self.beta_schedule.current = user["beta_current"]
        self._unique_seed = user.get("unique_seed")

    def load_merged(self, paths, streams=None):
        """Fill this shard from one or more checkpoints written by ``save`` for shards of any capacity, frame capacity
        and age limit (the same frame size and n-step gathering), merging them stream by stream (a0_ckpt_merge; the
        rule: ring_index.merge).  Every file's live records are taken oldest first; when this shard is smaller, the
        newest suffix stays.  Each kept record keeps its frames, action, reward, done, n-step window and priority bit
        for bit; record positions and frame seqs are renumbered, so this is not ``load``'s exact resume.
        ``streams=None`` takes every stream, file j's ids offset by j * S (S = 1 + the largest id of any file; file
        0's ids unchanged); otherwise one {old id: new id} dict per file names the streams taken.  max_p and the
        sampler's call counter are the maxima over the files; beta, the beta schedule's position and the
        draw-without-replacement seed come from file 0.  A stream whose observation stack is no longer in its file
        needs ``reset_streams`` before ``append_steps``.  Returns the files' user dicts.  Raises RuntimeError on a
        mismatched or corrupt file or colliding stream ids: a file rejected before the frames are decoded leaves the
        shard as it was, a failure while they are decoded leaves it empty.  CUDA graphs captured on the shard stay
        valid."""
        paths = [os.fsencode(os.fspath(p)) for p in paths]
        k = len(paths)
        map_old, map_new, map_len = stream_map_arrays(streams, k)
        cap = sum(os.path.getsize(p) for p in paths) if k else 0
        buf = C.create_string_buffer(max(1, min(cap, 1 << 16) * k))
        lens = np.zeros(k, dtype=np.int64)
        with torch.cuda.device(self.device):
            _lib.check(self.lib.a0_ckpt_merge(self.h, self.index.h, self._ex, (C.c_char_p * k)(*paths), k, map_old.ctypes.data,
                                              map_new.ctypes.data, map_len.ctypes.data, buf, len(buf), lens.ctypes.data,
                                              _lib.stream_ptr(self.device)), "a0_ckpt_merge")
        users, at = [], 0
        for n in lens.tolist():
            users.append(json.loads(buf.raw[at:at + n].decode()) if n else {})
            at += n
        self._apply_user(users[0])
        self.push_dynamic()
        return users

    @staticmethod
    def checkpoint_info(path):
        """Header and INDEX section of a checkpoint (a0_ckpt_info; the frames are not read): dict(N, NF, F, n_step,
        age_limit, live, sampleable, streams=[ids])."""
        lib = _lib.load()
        out = np.zeros(8, dtype=np.int64)
        ids = np.zeros(1 << 16, dtype=np.int64)
        _lib.check(lib.a0_ckpt_info(os.fsencode(os.fspath(path)), out.ctypes.data, ids.ctypes.data, len(ids)), "a0_ckpt_info")
        d = dict(zip(("N", "NF", "F", "n_step", "age_limit", "live", "sampleable"), out[:7].tolist()))
        d["streams"] = ids[:int(out[7])].tolist()
        return d

    def rng_seek(self, call):
        """Set the device-resident call counter of the sampler's own generator (stream-ordered)."""
        with torch.cuda.device(self.device):
            _lib.check(self.lib.a0_pt_rng_seek(self.h, int(call), _lib.stream_ptr(self.device)), "a0_pt_rng_seek")

    def set_priorities(self, ids, values):
        dev = self.device
        ids = torch.as_tensor(ids).to(device=dev, dtype=torch.int64).contiguous()
        values = torch.as_tensor(values).to(device=dev, dtype=torch.float32).contiguous()
        with torch.cuda.device(dev):
            _lib.check(self.lib.a0_pt_set(self.h, ids.data_ptr(), values.data_ptr(), ids.numel(),
                                          _lib.stream_ptr(dev)), "a0_pt_set")
