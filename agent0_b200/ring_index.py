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


# ------------------------------------------------------------------------------------------------------------------
# merging shard checkpoints into a shard of another shape (a0_ix_merge specification)
# ------------------------------------------------------------------------------------------------------------------
IX_MAGIC, IX_VERSION = 0x58493041, 1
REC_BYTES = SLOTS * 4 + 16           # one record of a RECORDS section: slots i32[8] + {reward f64, action|done i32, link i32}


def parse_index(blob):
    """The fields of an ``a0_ix_serialize`` blob (the INDEX section of a shard checkpoint) as a dict."""
    b = memoryview(bytes(blob))
    magic, ver = np.frombuffer(b[:8], dtype="<u4")
    assert magic == IX_MAGIC and ver == IX_VERSION, "not a ring index"
    N, NF, n, age, hq, tq, hfs, top = (int(x) for x in np.frombuffer(b[8:72], dtype="<i8"))
    at = 72
    d = dict(N=N, NF=NF, n=n, age_limit=age, head_q=hq, tail_q=tq, head_fs=hfs, top=top)
    d["fs_at_append"] = np.frombuffer(b[at:at + 8 * N], dtype="<i8").copy()
    at += 8 * N
    d["sampleable"] = np.frombuffer(b[at:at + N], dtype=np.uint8).astype(np.bool_)
    at += N
    i64 = lambda k: np.frombuffer(b[at:at + 8 * k], dtype="<i8").astype(np.int64)
    ns = int(i64(1)[0])
    at += 8
    streams = {}
    for _ in range(ns):
        sid, lp, ls, hs, s0, s1, s2, s3, k = (int(x) for x in i64(9))
        at += 72
        streams[sid] = dict(last_pos=lp, last_seq=ls, has_stack=bool(hs), stack=[s0, s1, s2, s3], pending=i64(k).tolist())
        at += 8 * k
    d["streams"] = streams
    nst = int(i64(1)[0])
    at += 8
    d["stale"] = set(i64(nst).tolist())
    return d


def serialize_index(ix, stacks=None):
    """``RingIndex`` state in the byte layout of ``a0_ix_serialize``; ``stacks``: stream -> i64[4] current stack."""
    stacks = stacks or {}
    out = [np.array([IX_MAGIC, IX_VERSION], dtype="<u4").tobytes(),
           np.array([ix.N, ix.NF, ix.n, ix.age_limit, ix.head_q, ix.tail_q, ix.head_fs, ix.top], dtype="<i8").tobytes(),
           np.asarray(ix.fs_at_append, dtype="<i8").tobytes(), np.asarray(ix.sampleable, dtype=np.uint8).tobytes()]
    ids = sorted(set(ix.streams) | set(stacks))
    out.append(np.array([len(ids)], dtype="<i8").tobytes())
    for sid in ids:
        st = ix.streams.get(sid, dict(last_pos=-1, last_seq=-1, pending=[]))
        stack = stacks.get(sid)
        words = [sid, st["last_pos"], st["last_seq"], 1 if stack is not None else 0] + \
            (list(stack) if stack is not None else [0, 0, 0, 0]) + [len(st["pending"])] + list(st["pending"])
        out.append(np.array(words, dtype="<i8").tobytes())
    stale = sorted(ix.stale)
    out.append(np.array([len(stale)] + stale, dtype="<i8").tobytes())
    return b"".join(out)


def empty_records(N):
    """RECORDS of a freshly reset shard: slots 0, info bytes 0xff (a0_rb_reset)."""
    slots = np.zeros((N, SLOTS), dtype=np.int32)
    info = np.full((N, 4), -1, dtype=np.int32)          # reward (2 words), action|done, link
    return slots, info


def apply_rec_meta(slots, info, meta):
    """What K1 writes for the records of one plan (a0_k1_write_record): slots, {reward, action|done, link} and the
    predecessor's link word.  Inside one plan no record is both written and named as a predecessor."""
    for mt in np.asarray(meta, dtype=np.int32):
        pos = int(mt[0])
        slots[pos] = mt[4:12]
        info[pos, 0:2] = mt[12:14]
        info[pos, 2] = mt[3]
        info[pos, 3] = mt[2]
        if mt[1] >= 0:
            info[int(mt[1]), 3] = pos


def stride_rule(meta, N, hint):
    """The successor stride a0_rb_ingest_plan keeps for K3 after one plan's records (csrc/a0_ingest.cu)."""
    stride = -1
    for mt in meta:
        if stride == 0:
            break
        if mt[1] < 0:
            continue
        dlt = int(mt[0]) - int(mt[1])
        if dlt <= 0:
            dlt += N
        stride = dlt if (stride < 0 or stride == dlt) else 0
    return stride if stride >= 0 else hint


def merge_stream_maps(sources, streams):
    """Rule 5: one {old id: new id} dict per file.  ``streams=None``: every stream, file j's ids offset by j * S
    (S = 1 + the largest id of any file).  Raises ValueError when two kept streams would share a new id."""
    present = [set(s["index"]["streams"]) | {t[0] for t in s.get("tails", ())} for s in sources]
    if streams is None:
        S = 1 + max((max(p) for p in present if p), default=-1)
        maps = [{sid: sid + j * S for sid in p} for j, p in enumerate(present)]
    else:
        assert len(streams) == len(sources), "one stream map per file"
        maps = [{int(a): int(b) for a, b in dict(m).items() if int(a) in p} for m, p in zip(streams, present)]
    seen = set()
    for m in maps:
        for new in m.values():
            if new in seen:
                raise ValueError(f"two kept streams would both become stream {new}")
            seen.add(new)
    return maps


def merge(target, sources, streams=None):
    """Specification of a0_ix_merge: fill the empty ``RingIndex`` ``target`` from k shard checkpoints.

    ``sources``: one dict per file, {index: parse_index(INDEX section), slots: i32[N,8], info: i32[N,4] (the RECORDS
    section), leaves: f32[N], tails: [(stream id, seq[8])] of its TAILS section}.  Returns dict(slots, info, leaves)
    of the target, ``stacks`` {new id: i64[4]}, ``placements`` i64[P,3] {file, source frame seq, target ring slot},
    ``record_map`` i64[R,3] {file, source position, target position or -1 when the target evicted it}, ``tails``
    [(new id, file, tail entry, seq[8])] in ascending new id, and ``stride_hint``.

      1. From each file the live records of the kept streams; a record's stream is found by walking the ``link`` words
         backwards from the stream's last record.
      2. Age head_q - 1 - q inside the file; all records oldest first, ties by file index.
      3. Fed to ``target.plan`` in chunks of ``target.max_chunk``.  A frame is (file, source seq); it reuses its newest
         target seq t when t is resident and next_fs - t < age_limit (ContentDeduper's rule), otherwise it gets the
         next new seq, in (record, slot) order.  The target's eviction rule keeps the newest suffix.
      4. A sampleable record keeps its source leaf; a record that was stale in its file (live, neither sampleable nor
         pending, or pending and in the stale set) enters the target's stale set, so it never becomes sampleable.
      5. Stream ids: see ``merge_stream_maps``.
      6. The kept streams' stacks whose frames are resident in their file are placed after the records (frames-only
         plans, ascending new id, the same reuse rule); TAILS entries take the newest target seq of each frame and
         are dropped when one of their frames is not resident in the target at the end.
    """
    k = len(sources)
    for s in sources:
        if s["index"]["n"] != target.n:
            raise ValueError(f"a file gathers n_step={s['index']['n']}, the target {target.n}")
    if target.head_q or target.head_fs or target.streams:
        raise ValueError("the target index is not empty")
    maps = merge_stream_maps(sources, streams)
    recs = []                          # (q - head_q, file, q, pos, stream, stale)
    for j, s in enumerate(sources):
        ix, slots, info = s["index"], s["slots"], s["info"]
        N, hq, tq = ix["N"], ix["head_q"], ix["tail_q"]
        seq_of = lambda pos: tq + (pos - tq % N) % N
        pred = {}
        for q in range(tq, hq):
            link = int(info[q % N, 3])
            if link >= 0:
                if link in pred:
                    raise ValueError(f"file {j}: two records link to record {link}")
                pred[link] = q % N
        pending = {p for st in ix["streams"].values() for p in st["pending"]}
        owner = {}
        for sid, st in ix["streams"].items():
            p = st["last_pos"] if st["last_seq"] >= tq else -1
            while p >= 0:
                if p in owner:
                    raise ValueError(f"file {j}: record {p} is reached twice")
                owner[p] = sid
                p = pred.get(p, -1)
        if len(owner) != hq - tq:
            raise ValueError(f"file {j}: {hq - tq - len(owner)} live records belong to no stream")
        for pos, sid in owner.items():
            if sid in maps[j]:
                q = seq_of(pos)
                stale = not ix["sampleable"][pos] and (q not in pending or q in ix["stale"])
                recs.append((q - hq, j, q, pos, maps[j][sid], stale))
    recs.sort()

    def src_seq(j, pos):
        ix = sources[j]["index"]
        lo = max(0, ix["head_fs"] - ix["NF"])
        return lo + (pos - lo % ix["NF"]) % ix["NF"]

    newest = {}                        # (file, source seq) -> newest target seq
    alloc = []                         # (target seq, file, source seq) in allocation order

    def resolve(idents, next_fs, hf):
        out = []
        for ident in idents:
            t = newest.get(ident)
            if t is None or t < hf - target.NF or next_fs - t >= target.age_limit:
                t = next_fs
                next_fs += 1
                newest[ident] = t
                alloc.append((t,) + ident)
            out.append(t)
        return out, next_fs

    N2 = target.N
    slots2, info2 = empty_records(N2)
    hint = 0
    tq_of = []                         # target seq of every merged record
    chunk = target.max_chunk
    for c0 in range(0, len(recs), chunk):
        part = recs[c0:c0 + chunk]
        m = len(part)
        hf = target.head_fs
        idents = [(r[1], src_seq(r[1], int(p))) for r in part for p in sources[r[1]]["slots"][r[3]]]
        fs, nxt = resolve(idents, hf, hf)
        fs8 = np.asarray(fs, dtype=np.int64).reshape(m, SLOTS)
        q0 = target.head_q
        target.stale.update(q0 + i for i, r in enumerate(part) if r[5])
        infos = [sources[r[1]]["info"][r[3]] for r in part]
        ad = np.array([int(x[2]) for x in infos], dtype=np.int64)
        reward = np.ascontiguousarray(np.array([x[0:2] for x in infos], dtype=np.int32)).view(np.float64).reshape(m)
        stream = np.array([r[4] for r in part], dtype=np.int64)
        p = target.plan(stream, fs8, np.arange(nxt - hf), ad & 0x7fffffff, reward, ad < 0)
        apply_rec_meta(slots2, info2, p.rec_meta)
        hint = stride_rule(p.rec_meta, N2, hint)
        tq_of.extend(range(q0, q0 + m))

    stacks = {}
    todo = []
    for j, s in enumerate(sources):
        ix = s["index"]
        lo = max(0, ix["head_fs"] - ix["NF"])
        for sid, st in ix["streams"].items():
            if sid in maps[j] and st["has_stack"] and all(lo <= f < ix["head_fs"] for f in st["stack"]):
                todo.append((maps[j][sid], j, st["stack"]))
    todo.sort(key=lambda x: x[0])
    per = max(1, 2 * chunk)            # streams per frames-only plan: at most 8 * max_chunk new frames
    for g0 in range(0, len(todo), per):
        hf = target.head_fs
        group = todo[g0:g0 + per]
        fs, nxt = resolve([(j, int(f)) for _, j, st in group for f in st], hf, hf)
        z = np.zeros(0, dtype=np.int64)
        target.plan(z, np.zeros((0, SLOTS), dtype=np.int64), np.arange(nxt - hf), z, z.astype(np.float64), z.astype(np.bool_))
        for i, (new, _, _) in enumerate(group):
            stacks[new] = np.asarray(fs[4 * i:4 * i + 4], dtype=np.int64)
            target.streams.setdefault(new, dict(last_pos=-1, last_seq=-1, pending=[]))

    final_lo = target.head_fs - target.NF
    tails = []
    for j, s in enumerate(sources):
        for e, (sid, seq8) in enumerate(s.get("tails", ())):
            if sid not in maps[j]:
                continue
            t = [newest.get((j, int(f)), -1) for f in seq8]
            if all(x >= 0 and x >= final_lo for x in t):
                tails.append((maps[j][sid], j, e, np.asarray(t, dtype=np.int64)))
    tails.sort(key=lambda x: x[0])

    leaves2 = np.zeros(N2, dtype=np.float32)
    rmap = []
    for r, q in zip(recs, tq_of):
        live = q >= target.tail_q
        dst = q % N2 if live else -1
        if live and target.sampleable[dst]:
            leaves2[dst] = sources[r[1]]["leaves"][r[3]]
        rmap.append((r[1], r[3], dst))
    place = np.array([(j, f, t % target.NF) for t, j, f in alloc if t >= final_lo], dtype=np.int64).reshape(-1, 3)
    return dict(slots=slots2, info=info2, leaves=leaves2, stacks=stacks, placements=place,
                record_map=np.array(rmap, dtype=np.int64).reshape(-1, 3), tails=tails, stride_hint=hint)


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

    def merge(self, sources, records, leaves, streams=None, tails=None):
        """a0_ix_merge into this (empty) index: ``sources`` NativeRingIndex of the files, ``records`` their RECORDS
        sections (bytes or u8/i32 arrays of N*48 bytes), ``leaves`` f32[N] each, ``streams`` as ``merge``, ``tails``
        one [(stream id, seq[8])] list per file (or None).  Returns what ``merge`` returns except ``stacks``
        (``get_stack`` reads them)."""
        C = self._C
        k = len(sources)
        recs = [np.frombuffer(bytes(r) if not isinstance(r, np.ndarray) else r.tobytes(), dtype=np.uint8) for r in records]
        lvs = [np.ascontiguousarray(x, dtype=np.float32) for x in leaves]
        for s, r, x in zip(sources, recs, lvs):
            assert r.size == s.N * REC_BYTES and x.size == s.N
        map_old, map_new, map_len = stream_map_arrays(streams, k)
        tails = tails or [[] for _ in range(k)]
        tcount = np.array([len(t) for t in tails], dtype=np.int64)
        tids = np.array([int(e[0]) for t in tails for e in t], dtype=np.int64)
        tseq = np.array([np.asarray(e[1], dtype=np.int64) for t in tails for e in t], dtype=np.int64).reshape(-1, SLOTS)
        ptrs = lambda arrs, T: (T * k)(*[C.cast(a.ctypes.data, T) for a in arrs])
        rec_out = np.zeros(self.N * REC_BYTES, dtype=np.uint8)
        leaf_out = np.zeros(self.N, dtype=np.float32)
        out = self._L.Merge()
        self._L.check(self.lib.a0_ix_merge(self.h, k, (C.c_void_p * k)(*[s.h.value for s in sources]), ptrs(recs, C.c_void_p),
                                           ptrs(lvs, C.c_void_p), map_old.ctypes.data, map_new.ctypes.data, map_len.ctypes.data,
                                           tcount.ctypes.data, tids.ctypes.data, tseq.ctypes.data, rec_out.ctypes.data,
                                           leaf_out.ctypes.data, C.byref(out)), "a0_ix_merge")
        arr = lambda p, n, w: np.ctypeslib.as_array(p, shape=(n * w,)).reshape(n, w).copy() if n else np.zeros((0, w), np.int64)
        tl = arr(out.tails, out.n_tail, 3 + SLOTS)
        slots = rec_out[:self.N * SLOTS * 4].view(np.int32).reshape(self.N, SLOTS).copy()
        info = rec_out[self.N * SLOTS * 4:].view(np.int32).reshape(self.N, 4).copy()
        return dict(slots=slots, info=info, leaves=leaf_out, placements=arr(out.place, out.n_place, 3),
                    record_map=arr(out.record_map, out.n_rec, 3),
                    tails=[(int(r[0]), int(r[1]), int(r[2]), r[3:].copy()) for r in tl], stride_hint=int(out.stride_hint))


def stream_map_arrays(streams, k):
    """(map_old, map_new, map_len) of the C ABI for ``streams`` = None (every stream of every file, rule 5) or one
    {old id: new id} dict per file."""
    if streams is None:
        return np.zeros(1, np.int64), np.zeros(1, np.int64), np.full(k, -1, dtype=np.int64)
    assert len(streams) == k, "one stream map per file"
    old = [int(a) for m in streams for a in dict(m)]
    new = [int(b) for m in streams for b in dict(m).values()]
    return (np.array(old + [0], dtype=np.int64), np.array(new + [0], dtype=np.int64),
            np.array([len(dict(m)) for m in streams], dtype=np.int64))
