"""Host-side index of the HBM replay shard (pure numpy; no CUDA needed, so it is unit-tested on CPU).

The reference keeps every transition as a self-contained 8-frame blob in a host deque
(agent0/deepq/replay.py:18, agent0/deepq/agent.py:78-81).  Here frames live once in an HBM frame
ring and a transition is a 48-byte *record* that names the 8 frame slots of its two stacks.  This
class decides, for every appended transition, which incoming frames are new, where they go, which
records become sampleable and which must be evicted; the CUDA kernels (K1/K2b) only execute the
plan it emits.  All quantities are sequence numbers (monotone int64); ring position = seq % capacity.

Rules (DESIGN.md, "validity"):
  * a frame seq f is resident while f >= head_fs - NF;
  * a record is evicted when its ring slot is reused, or when frames it may reference are about to
    be overwritten.  The test is conservative and monotone, so the live records are always the
    contiguous seq window [tail_q, head_q):  evict q  iff  fs_at_append[q] - age_limit < head_fs - NF;
  * a matched (de-duplicated) frame older than ``age_limit`` frames is stored again, which makes the
    bound above valid for any stream (static screens included);
  * with n-step gathering a record becomes sampleable when its (n-1)-th successor in the same
    stream has been appended (the reference's actor emits entry k-n+1 at step k, agent.py:64-73).
"""
from __future__ import annotations

import numpy as np

SLOTS = 8
META_I32 = 14


class AppendPlan:
    """What one append must do on the device."""
    __slots__ = ("new_frame_src", "new_frame_pos", "rec_meta", "marks", "count")

    def __init__(self, new_frame_src, new_frame_pos, rec_meta, marks, count):
        self.new_frame_src = new_frame_src    # int64 [n_new] index into the caller's flat frame list
        self.new_frame_pos = new_frame_pos    # int32 [n_new] frame-ring positions
        self.rec_meta = rec_meta              # int32 [m, 14]  (a0_rb_append layout)
        self.marks = marks                    # int32 [k]  >=0 newly sampleable pos, <0 ~pos evicted
        self.count = count


class RingIndex:
    def __init__(self, rec_capacity, frame_capacity, n_step=1, age_limit=None):
        assert n_step >= 1
        self.N, self.NF, self.n = int(rec_capacity), int(frame_capacity), int(n_step)
        self.age_limit = int(age_limit) if age_limit is not None else max(8, min(32768, self.NF // 8))
        assert self.NF > 2 * self.age_limit, "frame ring too small for the age limit"
        self.head_q = 0           # records appended so far
        self.tail_q = 0           # oldest live record
        self.head_fs = 0          # frames allocated so far
        self.top = 0              # sampleable records (the reference's `top`, replay.py:48)
        self.fs_at_append = np.zeros(self.N, dtype=np.int64)
        self.sampleable = np.zeros(self.N, dtype=np.bool_)
        self.streams = {}         # stream id -> dict(last_pos, last_seq, pending[list of seq])
        self.stale = set()        # seqs whose own frames were older than age_limit when appended

    # ------------------------------------------------------------------ limits
    @property
    def max_chunk(self):
        """Largest number of transitions one plan may hold (a plan must not overwrite itself)."""
        return max(1, min(self.N // 2, (self.NF - 2 * self.age_limit) // (2 * SLOTS)))

    def frame_resident(self, fs):
        return fs >= self.head_fs - self.NF

    # ------------------------------------------------------------------ planning
    def plan(self, stream, fs8, new_src, action, reward, done):
        """Commit m transitions whose 8 frame seqs are already resolved.

        stream i64[m]; fs8 i64[m,8] frame sequence numbers (new ones were numbered from
        ``self.head_fs`` upwards in increasing order); new_src i64[n_new]: for each new frame, in
        seq order, its index in the caller's flat frame array.  Returns an AppendPlan.
        """
        m = len(stream)
        assert m <= self.max_chunk, "append too large for the ring: split it"
        n_new = len(new_src)
        N, NF, n = self.N, self.NF, self.n
        q0 = self.head_q
        seq = q0 + np.arange(m, dtype=np.int64)
        pos = (seq % N).astype(np.int32)
        new_head_fs = self.head_fs + n_new
        new_head_q = q0 + m
        marks = []
        # a record whose frames are already older than the age limit (an idle stream that resumes)
        # can never be a sampling start: the eviction bound below would not cover it
        too_old = (self.head_fs - np.asarray(fs8, dtype=np.int64).min(axis=1)) > self.age_limit
        if too_old.any():
            self.stale.update(seq[too_old].tolist())

        # ---- evictions (prefix of the live window) --------------------------------------------
        thr = new_head_fs - NF
        while self.tail_q < q0:
            hi = min(q0, self.tail_q + 4 * m + 64)
            w = np.arange(self.tail_q, hi, dtype=np.int64)
            wp = w % N
            ev = (w < new_head_q - N) | (self.fs_at_append[wp] - self.age_limit < thr)
            k = int(ev.sum())                  # monotone: the evicted ones are a prefix
            if k == 0:
                break
            gone = wp[:k]
            self.top -= int(self.sampleable[gone].sum())
            self.sampleable[gone] = False
            marks.append(~gone.astype(np.int32))
            self.tail_q += k
            if k < len(w):
                break

        # ---- links and sampleability, stream by stream --------------------------------------------
        link_from = np.full(m, -1, dtype=np.int32)
        link_to = np.full(m, -1, dtype=np.int32)
        order = np.argsort(stream, kind="stable")
        ss = stream[order]
        bounds = np.flatnonzero(np.r_[True, ss[1:] != ss[:-1], True])
        newly = []
        for gi in range(len(bounds) - 1 if m else 0):
            idx = order[bounds[gi]:bounds[gi + 1]]          # batch indices of this stream, in order
            sid = int(ss[bounds[gi]])
            st = self.streams.get(sid)
            if st is None:
                st = self.streams[sid] = dict(last_pos=-1, last_seq=-1, pending=[])
            if st["last_seq"] >= max(self.tail_q, q0 - N):   # predecessor still live
                link_from[idx[0]] = st["last_pos"]
            link_to[idx[:-1]] = pos[idx[1:]]
            if n == 1:
                newly.append(seq[idx])
            else:
                combined = np.concatenate((np.asarray(st["pending"], dtype=np.int64), seq[idx]))
                ready = len(combined) - (n - 1)
                if ready > 0:
                    newly.append(combined[:ready])
                st["pending"] = combined[max(ready, 0):].tolist()
            st["last_pos"], st["last_seq"] = int(pos[idx[-1]]), int(seq[idx[-1]])
        self.fs_at_append[pos] = self.head_fs      # frames allocated before this plan (monotone key)
        self.head_q, self.head_fs = new_head_q, new_head_fs
        if newly:
            ready = np.concatenate(newly)
            ready = ready[ready >= self.tail_q]          # evicted before it ever became sampleable
            if self.stale:
                keep = np.array([int(r) not in self.stale for r in ready], dtype=np.bool_)
                self.stale = {r for r in self.stale if r >= self.tail_q and r not in set(ready.tolist())}
                ready = ready[keep]
            rp = (ready % N).astype(np.int32)
            self.sampleable[rp] = True
            self.top += len(rp)
            marks.append(rp)

        # ---- record metadata --------------------------------------------------------------------
        meta = np.empty((m, META_I32), dtype=np.int32)
        meta[:, 0] = pos
        meta[:, 1] = link_from
        meta[:, 2] = link_to
        meta[:, 3] = (np.asarray(action, dtype=np.int64) & 0x7fffffff).astype(np.int32) | \
            (np.asarray(done, dtype=np.bool_).astype(np.int32) << 31)
        meta[:, 4:12] = (np.asarray(fs8, dtype=np.int64) % NF).astype(np.int32)
        meta[:, 12:14] = np.ascontiguousarray(np.asarray(reward, dtype=np.float64)).view(np.int32).reshape(m, 2)
        new_pos = ((self.head_fs - n_new + np.arange(n_new, dtype=np.int64)) % NF).astype(np.int32)
        marks = np.concatenate(marks).astype(np.int32) if marks else np.zeros(0, dtype=np.int32)
        return AppendPlan(np.asarray(new_src, dtype=np.int64), new_pos, meta, marks, m)

    # ------------------------------------------------------------------ structural (native) ingest
    def resolve_shift(self, stream, n_new, last4):
        """Frame seqs for transitions described structurally: the observation stack of each
        transition is the stream's current stack and the next stack is that stack shifted by
        ``n_new`` (0..4) new frames.  ``stream`` i64[m] in commit order, ``last4`` dict
        stream -> i64[4] current stack seqs (updated in place).  New frames are numbered in
        (transition, frame) order from head_fs.  Returns fs8 i64[m,8]."""
        m = len(stream)
        n_new = np.asarray(n_new, dtype=np.int64)
        off = self.head_fs + np.concatenate(([0], np.cumsum(n_new)[:-1])).astype(np.int64)
        fs8 = np.empty((m, SLOTS), dtype=np.int64)
        order = np.argsort(stream, kind="stable")
        ss = stream[order]
        bounds = np.flatnonzero(np.r_[True, ss[1:] != ss[:-1], True])
        for gi in range(len(bounds) - 1 if m else 0):
            idx = order[bounds[gi]:bounds[gi + 1]]
            sid = int(ss[bounds[gi]])
            c = n_new[idx]
            # the stream's frame list: current stack, then its new frames step by step
            reps = np.repeat(off[idx], c) + (np.arange(c.sum()) - np.repeat(np.cumsum(c) - c, c))
            L = np.concatenate((last4[sid], reps))
            end = np.cumsum(c)                      # frames of the stream consumed after each step
            ar = np.arange(4)
            fs8[idx, :4] = L[(end - c)[:, None] + ar]
            fs8[idx, 4:] = L[end[:, None] + ar]
            last4[sid] = L[-4:].copy()
        return fs8


class ContentDeduper:
    """Content-based frame de-duplication for the reference-compatible ingest.

    The reference's entries are self-contained 8-frame blobs (agent0/deepq/agent.py:78-81), 7 of
    which normally repeat frames of the same env's previous entry.  A frame is matched, by 64-bit
    hash and then by full byte comparison (so a match is always bit-exact), against the 8 frames
    of the stream's previous entry and the earlier frames of the same entry; unmatched frames are
    new.  Matches older than the index's age limit are stored again (see RingIndex)."""

    _SEED = 0x9E3779B97F4A7C15

    def __init__(self, index, frame_bytes):
        assert frame_bytes % 8 == 0
        self.ix, self.F = index, frame_bytes
        self.mult = (np.arange(1, frame_bytes // 8 + 1, dtype=np.uint64) * np.uint64(self._SEED)) | np.uint64(1)
        self.tail = {}     # stream -> (u8[8,F] frames, i64[8] seqs, u64[8] hashes) of its last entry

    def resolve(self, streams, frames):
        """frames u8[m,8,F] (C-contiguous).  Returns fs8 i64[m,8] and new_src i64[n_new] (flat
        indices t*8+j of the frames that must be stored, in allocation order)."""
        m = len(streams)
        ix = self.ix
        hashes = (frames.reshape(m, 8, self.F // 8, 8).view(np.uint64)[..., 0] * self.mult).sum(axis=2)
        fs8 = np.empty((m, 8), dtype=np.int64)
        new_src = []
        next_fs = ix.head_fs
        for t in range(m):
            sid = int(streams[t])
            prev = self.tail.get(sid)
            for j in range(8):
                hit = -1
                if prev is not None:
                    pf, pfs, ph = prev
                    for c in np.flatnonzero(ph == hashes[t, j]):
                        if next_fs - pfs[c] < ix.age_limit and ix.frame_resident(pfs[c]) and \
                                np.array_equal(pf[c], frames[t, j]):
                            hit = int(pfs[c])
                            break
                if hit < 0:
                    for c in np.flatnonzero(hashes[t, :j] == hashes[t, j]):
                        if np.array_equal(frames[t, c], frames[t, j]):
                            hit = int(fs8[t, c])
                            break
                if hit < 0:
                    hit = next_fs
                    next_fs += 1
                    new_src.append(t * 8 + j)
                fs8[t, j] = hit
            prev = self.tail[sid] = (frames[t], fs8[t].copy(), hashes[t])
        return fs8, np.asarray(new_src, dtype=np.int64)

    def detach(self, streams):
        """Take private copies of the stream tails (the caller may reuse its buffers)."""
        for sid in set(int(s) for s in streams):
            f, s_, h_ = self.tail[sid]
            self.tail[sid] = (f.copy(), s_, h_.copy())


class NativeContentDeduper:
    """ContentDeduper's rule in C++ (csrc/a0_ingest.cu: a0_dd_resolve) -- the one ``ReplayDataset.extend``
    uses: 1280 reference entries (72 MB) resolve in ~20 ms instead of ~260 ms of numpy.  The Python class
    above stays as the executable specification (tests/test_ring_index.py requires identical output)."""

    def __init__(self, index, frame_bytes):
        import ctypes as C

        from . import _lib
        assert isinstance(index, NativeRingIndex), "the native deduper reads the native index"
        self._C, self._L, self.ix, self.F = C, _lib, index, int(frame_bytes)
        self.lib = _lib.load()
        h = C.c_void_p()
        _lib.check(self.lib.a0_dd_create(C.byref(h), self.F), "a0_dd_create")
        self.h = h

    def __del__(self):
        try:
            if getattr(self, "h", None) is not None and self.h.value:
                self.lib.a0_dd_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def resolve(self, streams, frames):
        """frames u8[m,8,F] (C-contiguous).  Returns fs8 i64[m,8] and new_src i64[n_new]."""
        streams = np.ascontiguousarray(streams, dtype=np.int64)
        frames = np.ascontiguousarray(frames, dtype=np.uint8)
        m = len(streams)
        assert frames.size == m * SLOTS * self.F
        fs8 = np.empty((m, SLOTS), dtype=np.int64)
        new_src = np.empty(m * SLOTS, dtype=np.int64)
        n_new = self._C.c_int32(0)
        self._L.check(self.lib.a0_dd_resolve(self.h, self.ix.h, streams.ctypes.data, frames.ctypes.data, m, fs8.ctypes.data,
                                             new_src.ctypes.data, self._C.byref(n_new)), "a0_dd_resolve")
        return fs8, new_src[:n_new.value].copy()

    def detach(self, streams):
        """No-op: a0_dd_resolve already took private copies of the stream tails."""


def stack_delta(prev_stack, next_stack):
    """Smallest k in 0..4 such that next_stack[:4-k] == prev_stack[k:] (how many new frames a
    vector-env step brought).  Stacks are uint8 [E,4,...]; returns int64 [E]."""
    E = prev_stack.shape[0]
    p = prev_stack.reshape(E, 4, -1)
    q = next_stack.reshape(E, 4, -1)
    k = np.full(E, 4, dtype=np.int64)
    for cand in (3, 2, 1, 0):
        ok = (q[:, :4 - cand] == p[:, cand:]).all(axis=(1, 2))
        k = np.where(ok, cand, k)
    return k


class NativeRingIndex:
    """The same index, implemented in C++ inside libagent0_b200.so (csrc/a0_ingest.cu) so that an
    append costs microseconds of host time instead of ~0.6 ms of numpy; this is the one
    ``ReplayDataset`` uses.  ``RingIndex`` above stays as the executable specification:
    tests/test_ring_index.py drives both with the same streams and requires identical plans."""

    def __init__(self, rec_capacity, frame_capacity, n_step=1, age_limit=None):
        import ctypes as C

        from . import _lib
        self._C, self._L = C, _lib
        self.lib = _lib.load()
        h = C.c_void_p()
        _lib.check(self.lib.a0_ix_create(C.byref(h), int(rec_capacity), int(frame_capacity), int(n_step),
                                         -1 if age_limit is None else int(age_limit)), "a0_ix_create")
        self.h = h
        self._state = np.zeros(_lib.IX_STATE_WORDS, dtype=np.int64)
        self._refresh()
        st = self._state
        self.N, self.NF, self.n = int(st[_lib.IX_REC_CAPACITY]), int(st[_lib.IX_FRAME_CAPACITY]), int(st[_lib.IX_NSTEP])
        self.age_limit, self.max_chunk = int(st[_lib.IX_AGE_LIMIT]), int(st[_lib.IX_MAX_CHUNK])
        buf = (C.c_uint8 * self.N).from_address(self.lib.a0_ix_sampleable(h))
        self.sampleable = np.frombuffer(buf, dtype=np.uint8).view(np.bool_)      # live view of host state
        self._plan = _lib.Plan()

    def __del__(self):
        try:
            if getattr(self, "h", None) is not None and self.h.value:
                self.lib.a0_ix_destroy(self.h)
                self.h = None
        except Exception:
            pass

    def _refresh(self):
        self.lib.a0_ix_state(self.h, self._state.ctypes.data)

    head_q = property(lambda self: (self._refresh(), int(self._state[0]))[1])
    tail_q = property(lambda self: (self._refresh(), int(self._state[1]))[1])
    head_fs = property(lambda self: (self._refresh(), int(self._state[2]))[1])
    top = property(lambda self: (self._refresh(), int(self._state[3]))[1])

    def frame_resident(self, fs):
        return fs >= self.head_fs - self.NF

    def set_stack(self, stream, seq4):
        seq4 = np.ascontiguousarray(seq4, dtype=np.int64)
        self._L.check(self.lib.a0_ix_set_stack(self.h, int(stream), seq4.ctypes.data), "a0_ix_set_stack")

    def get_stack(self, stream):
        out = np.empty(4, dtype=np.int64)
        return out if self.lib.a0_ix_get_stack(self.h, int(stream), out.ctypes.data) == 0 else None

    def has_stack(self, stream):
        return self.get_stack(stream) is not None

    def resolve_shift(self, stream, n_new, last4=None):
        """``last4`` (dict stream -> i64[4]) is honoured for interface parity with RingIndex: its
        stacks are pushed into the native index before and read back after the call."""
        stream = np.ascontiguousarray(stream, dtype=np.int64)
        n_new = np.ascontiguousarray(n_new, dtype=np.int64)
        m = len(stream)
        if last4 is not None:
            for sid in set(stream.tolist()):
                self.set_stack(sid, last4[sid])
        fs8 = np.empty((m, SLOTS), dtype=np.int64)
        self._L.check(self.lib.a0_ix_resolve_shift(self.h, stream.ctypes.data, n_new.ctypes.data, m, fs8.ctypes.data),
                      "a0_ix_resolve_shift")
        if last4 is not None:
            for sid in set(stream.tolist()):
                last4[sid] = self.get_stack(sid)
        return fs8

    def serialize(self):
        """The whole index state as bytes (a0_ix_serialize; the INDEX section of a shard checkpoint)."""
        n = self._C.c_int64(0)
        self.lib.a0_ix_serialize(self.h, None, 0, self._C.byref(n))
        buf = (self._C.c_uint8 * n.value)()
        self._L.check(self.lib.a0_ix_serialize(self.h, buf, n.value, self._C.byref(n)), "a0_ix_serialize")
        return bytes(buf)

    def deserialize(self, blob):
        """Replace the state with ``serialize()`` output of an index with the same parameters (a0_ix_deserialize)."""
        blob = bytes(blob)
        self._L.check(self.lib.a0_ix_deserialize(self.h, blob, len(blob)), "a0_ix_deserialize")

    def plan_native(self, stream, fs8, n_new, action, reward, done):
        """a0_ix_plan; returns the ctypes a0_plan_t (arrays owned by the index until its next call)."""
        stream = np.ascontiguousarray(stream, dtype=np.int64)
        fs8 = np.ascontiguousarray(fs8, dtype=np.int64)
        action = np.ascontiguousarray(action, dtype=np.int64)
        reward = np.ascontiguousarray(reward, dtype=np.float64)
        done = np.ascontiguousarray(done, dtype=np.bool_).view(np.uint8)
        m = len(stream)
        self._L.check(self.lib.a0_ix_plan(self.h, stream.ctypes.data, fs8.ctypes.data, m, int(n_new), action.ctypes.data,
                                          reward.ctypes.data, done.ctypes.data, self._C.byref(self._plan)), "a0_ix_plan")
        return self._plan

    def plan(self, stream, fs8, new_src, action, reward, done):
        new_src = np.asarray(new_src, dtype=np.int64)
        p = self.plan_native(stream, fs8, len(new_src), action, reward, done)
        arr = lambda ptr, k: np.ctypeslib.as_array(ptr, shape=(k,)).copy() if k else np.zeros(0, dtype=np.int32)
        return AppendPlan(new_src, arr(p.new_frame_pos, p.n_new), arr(p.rec_meta, p.m * META_I32).reshape(p.m, META_I32),
                          arr(p.marks, p.n_marks), p.m)
