"""Transitions from actors in their own processes into the learner's shard: a device inbox (K9, a0_inbox.cu).

The reference's actor nodes return 1280 transitions to the trainer node over RPC at the end of every ``Actor.sample``
(agent0/deepq/launch.py:45-63).  Here the learner owns a ``TransitionInbox``: a device region with one lane per actor
process, each lane a short ring of slots.  A ``TransitionWriter`` in the actor's process (CUDA IPC; on the same GPU or
a peer GPU) packs vector steps into page-locked staging and commits a slot with one kernel that never waits; the
learner's ``drain`` copies the committed slots' metadata to the host (one synchronise), feeds them to the shard with the
native ingest -- the frames are read by K1 straight from the slot -- and releases the slots.  No frame crosses the
host, and nothing runs on the learner's GIL but the ingest calls themselves.

The shard a drain builds is bit for bit the one in-process ``ReplayDataset.append_vector_step`` calls would have built
in the same order, stream ids offset by ``lane * streams_per_lane``: every vector step is one ``append_steps`` call, as
in-process.  (One call for a run of steps would not do: the ring index stamps all records of a call with the frame
head at its start, and the age-limit eviction reads that stamp.)
"""
from __future__ import annotations

import ctypes as C
import time
from collections import namedtuple

import numpy as np
import torch

from . import _lib
from .ring_index import stack_delta

LAYOUT_FIELDS = ("step_count", "step_reset", "stream", "n_new", "action", "reward", "done", "frames", "slot_bytes",
                 "lane_bytes", "region_bytes", "scan_meta", "scan_bytes", "ctl_bytes", "lane_header_bytes")
_ARRAYS = (("step_count", np.int64), ("step_reset", np.uint8), ("stream", np.int64), ("n_new", np.int64),
           ("action", np.int64), ("reward", np.float64), ("done", np.uint8))

Step = namedtuple("Step", ["reset", "stream", "n_new", "action", "reward", "done", "frame_off", "n_frames"])
Step.__doc__ = """One vector step of a slot: ``reset`` (its streams start here: their 4-frame stacks come first), the
per-transition arrays (local stream ids), and where its frames sit in the slot's frames."""


def slot_layout(slot_transitions, slot_frames, frame_bytes, lanes=1, slots=1):
    """The byte offsets of the region and of a slot (a0_tx_layout; no GPU needed) as a dict of LAYOUT_FIELDS."""
    out = np.zeros(len(LAYOUT_FIELDS), dtype=np.int64)
    _lib.check(_lib.load().a0_tx_layout(int(slot_transitions), int(slot_frames), int(frame_bytes), int(lanes), int(slots),
                                        out.ctypes.data), "a0_tx_layout")
    return dict(zip(LAYOUT_FIELDS, out.tolist()))


def _arrays(buf, layout, T):
    return {k: buf[layout[k]:layout[k] + T * np.dtype(dt).itemsize].view(dt) for k, dt in _ARRAYS}


class SlotPacker:
    """Packs vector steps into a buffer with a slot's layout (``buf``: u8 numpy array of at least ``slot_bytes``; the
    writer's page-locked staging).  Host code only."""

    def __init__(self, buf, layout, slot_transitions, slot_frames, frame_bytes):
        self.T, self.SF, self.F = int(slot_transitions), int(slot_frames), int(frame_bytes)
        self.buf = buf
        self.a = _arrays(buf, layout, self.T)
        self.frames = buf[layout["frames"]:layout["frames"] + self.SF * self.F].reshape(self.SF, self.F)
        self.frames_off = layout["frames"]
        self.clear()

    def clear(self):
        self.n_transitions = self.n_steps = self.n_frames = 0

    def fits(self, E, n_frames):
        return self.n_transitions + E <= self.T and self.n_steps + 1 <= self.T and self.n_frames + n_frames <= self.SF

    def add(self, reset, stream, n_new, action, reward, done, frames):
        """One vector step: E transitions and their frames (u8 [n, F]: the E stacks of a reset step, then the new frames
        in transition order)."""
        E, nf = len(stream), len(frames)
        assert self.fits(E, nf)
        t, s, f = self.n_transitions, self.n_steps, self.n_frames
        a = self.a
        a["step_count"][s] = E
        a["step_reset"][s] = 1 if reset else 0
        a["stream"][t:t + E] = stream
        a["n_new"][t:t + E] = n_new
        a["action"][t:t + E] = action
        a["reward"][t:t + E] = reward
        a["done"][t:t + E] = np.asarray(done, dtype=np.bool_)
        self.frames[f:f + nf] = frames
        self.n_transitions, self.n_steps, self.n_frames = t + E, s + 1, f + nf
        self.buf[:24].view(np.int64)[:] = (self.n_transitions, self.n_steps, self.n_frames)

    def nbytes(self):
        """Bytes of the buffer a commit copies: header, metadata and the frames packed so far."""
        return self.frames_off + self.n_frames * self.F


def parse_slot(meta, layout, slot_transitions, slot_frames, streams_per_lane, where="slot"):
    """The vector steps of a slot's header and metadata (``meta``: u8 array, at least ``layout['frames']`` bytes), after
    checking every field against the slot's capacity; a malformed slot raises RuntimeError naming ``where``."""
    T, SF, E_lane = int(slot_transitions), int(slot_frames), int(streams_per_lane)

    def bad(why):
        raise RuntimeError(f"transition inbox: {where} is malformed: {why}")

    n_t, n_s, n_f = (int(x) for x in meta[:24].view(np.int64))
    if not 1 <= n_t <= T:
        bad(f"{n_t} transitions outside [1, {T}]")
    if not 1 <= n_s <= n_t:
        bad(f"{n_s} vector steps outside [1, {n_t}]")
    if not 0 <= n_f <= SF:
        bad(f"{n_f} frames outside [0, {SF}]")
    a = _arrays(meta, layout, T)
    count, reset = a["step_count"][:n_s], a["step_reset"][:n_s]
    stream, n_new, done = a["stream"][:n_t], a["n_new"][:n_t], a["done"][:n_t]
    if count.min() < 1 or count.max() > E_lane:
        bad(f"a vector step of {int(count.min() if count.min() < 1 else count.max())} transitions, outside [1, {E_lane}]")
    if int(count.sum()) != n_t:
        bad(f"the vector steps hold {int(count.sum())} transitions, the header {n_t}")
    if reset.max() > 1:
        bad(f"reset flag {int(reset.max())}")
    if stream.min() < 0 or stream.max() >= E_lane:
        bad(f"stream id {int(stream.min() if stream.min() < 0 else stream.max())} outside [0, {E_lane})")
    if n_new.min() < 0 or n_new.max() > 4:
        bad(f"n_new {int(n_new.min() if n_new.min() < 0 else n_new.max())} outside [0, 4]")
    if done.max() > 1:
        bad(f"done flag {int(done.max())}")
    want = 4 * int(count[reset == 1].sum()) + int(n_new.sum())
    if want != n_f:
        bad(f"{n_f} frames where the resets and n_new need {want}")
    steps, t, f = [], 0, 0
    for k, r in zip(count.tolist(), reset.tolist()):
        sl = slice(t, t + k)
        nf = 4 * k * r + int(n_new[sl].sum())
        steps.append(Step(bool(r), stream[sl], n_new[sl], a["action"][sl], a["reward"][sl], done[sl], f, nf))
        t, f = t + k, f + nf
    return steps


class TransitionInbox:
    """The learner's side: ``lanes`` lanes of ``slots`` slots next to ``replay`` (a native_nstep=True shard).  Lane ``l``
    owns the shard's streams [l * E, (l + 1) * E), E = ``cfg.actor.num_envs``.  The default slot holds one
    ``ShardActor.sample`` call: num_envs * sample_steps transitions and max(2 * transitions + 4 * num_envs,
    8 * num_envs) frames.  A slot must take any one vector step, so ``slot_transitions`` >= E and ``slot_frames`` >= 8E
    (a writer's first step carries the E reset stacks and up to 4 new frames per stream); a smaller one is refused."""

    def __init__(self, replay, lanes, slots=4, slot_transitions=None, slot_frames=None):
        cfg = replay.cfg
        self.replay, self.lib, self.device = replay, _lib.load(), replay.device
        self.E = int(cfg.actor.num_envs)
        self.lanes, self.slots = int(lanes), int(slots)
        self.T = int(slot_transitions or self.E * int(cfg.actor.sample_steps))
        self.SF = int(slot_frames or max(2 * self.T + 4 * self.E, 8 * self.E))
        if self.T < self.E:
            raise ValueError(f"slot_transitions {self.T} is below one vector step of {self.E} streams")
        if self.SF < 8 * self.E:
            raise ValueError(f"slot_frames {self.SF} is below the {8 * self.E} frames a writer's first vector step of "
                             f"{self.E} streams can carry")
        self.F = replay.F
        self.layout = slot_layout(self.T, self.SF, self.F, self.lanes, self.slots)
        h = C.c_void_p()
        _lib.check(self.lib.a0_tx_create(C.byref(h), self.lanes, self.slots, self.T, self.SF, self.F, self.E,
                                         replay.n_gather, self.device.index), "a0_tx_create")
        self._h = h
        L = self.layout
        self._scan = np.ctypeslib.as_array((C.c_uint8 * L["scan_bytes"]).from_address(self.lib.a0_tx_scan_host(h)))
        self._frames = [[_lib.device_view(self.lib.a0_tx_slot_frames(h, l, s), (self.SF, self.F), "|u1", self.device, owner=self)
                         for s in range(self.slots)] for l in range(self.lanes)]

    def handle(self, lane):
        """What an actor process opens a ``TransitionWriter`` with (picklable): the IPC handle, the slot layout, the lane
        and the PCI bus id of the learner's GPU."""
        if not 0 <= lane < self.lanes:
            raise ValueError(f"lane {lane} outside [0, {self.lanes})")
        buf = (C.c_uint8 * 64)()
        _lib.check(self.lib.a0_tx_handle(self._h, buf), "a0_tx_handle")
        return dict(ipc=bytes(buf), lane=int(lane), lanes=self.lanes, slots=self.slots, slot_transitions=self.T,
                    slot_frames=self.SF, frame_bytes=self.F, frame_shape=tuple(self.replay.frame_shape),
                    streams_per_lane=self.E, n_gather=self.replay.n_gather, layout=dict(self.layout),
                    pci_bus_id=_lib.pci_bus_id(self.device.index))

    def drain(self):
        """Ingests every committed slot of every lane (up to ``slots`` per lane) into the shard and releases them.
        Returns the number of transitions ingested.  Every slot is validated before any is ingested: a malformed one
        raises RuntimeError naming its lane and slot, nothing of the drain is ingested, and the lane stays blocked."""
        rp, lib, dev, L = self.replay, self.lib, self.device, self.layout
        S, E = self.slots, self.E
        with torch.cuda.device(dev):
            _lib.check(lib.a0_tx_scan(self._h, S, _lib.stream_ptr(dev)), "a0_tx_scan")
            torch.cuda.current_stream(dev).synchronize()
        head = self._scan[:32 * self.lanes].view(np.int64).reshape(self.lanes, 4)
        todo = []
        for l in range(self.lanes):
            consumed, committed, taken = (int(x) for x in head[l, :3])
            if not 0 <= committed - consumed <= S:
                raise RuntimeError(f"transition inbox: lane {l} is malformed: committed {committed} - consumed {consumed} "
                                   f"outside [0, {S}]")
            for j in range(taken):
                at = L["scan_meta"] + (l * S + j) * L["frames"]
                slot = (consumed + j) % S
                todo.append((l, slot, parse_slot(self._scan[at:at + L["frames"]], L, self.T, self.SF, E,
                                                 where=f"lane {l}, slot {slot}")))
        n = 0
        for l, slot, steps in todo:
            frames = self._frames[l][slot]
            for st in steps:
                streams = st.stream + l * E
                f = st.frame_off
                if st.reset:
                    k = 4 * len(streams)
                    rp.reset_streams(streams, frames[f:f + k])
                    f += k
                rp.append_steps(streams, st.n_new, frames[f:st.frame_off + st.n_frames], st.action, st.reward, st.done)
                n += len(streams)
        if todo:
            with torch.cuda.device(dev):
                _lib.check(lib.a0_tx_release(self._h, _lib.stream_ptr(dev)), "a0_tx_release")
        return n

    def unclaim(self, lane):
        """Frees the lane of a writer that died, so that a new writer can open it.  Slots that writer committed are
        still drained; one it left half-written is never seen."""
        _lib.check(self.lib.a0_tx_unclaim(self._h, int(lane)), "a0_tx_unclaim")

    def region(self):
        """TEST HOOK: the whole region as a u8 device view (control block, lane words, slots)."""
        return _lib.device_view(self.lib.a0_tx_ctl(self._h), (self.layout["region_bytes"],), "|u1", self.device, owner=self)

    def lane_words(self, lane):
        """TEST HOOK: lane ``lane``'s {claimed, committed, consumed} as i64 device views (each on its own 128-B line)."""
        at = self.layout["ctl_bytes"] + lane * self.layout["lane_bytes"]
        return self.region()[at:at + 384].view(torch.int64)[::16]

    def slot_bytes(self, lane, slot):
        """TEST HOOK: the bytes of one slot as a u8 device view."""
        L = self.layout
        at = L["ctl_bytes"] + lane * L["lane_bytes"] + L["lane_header_bytes"] + slot * L["slot_bytes"]
        return self.region()[at:at + L["slot_bytes"]]

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.a0_tx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class TransitionWriter:
    """The actor's side: appends vector steps to one lane of a ``TransitionInbox``.

    ``handle``: ``TransitionInbox.handle(lane)`` from another process (mapped with CUDA IPC; from another GPU of the node
    the stores go over NVLink), or the ``TransitionInbox`` itself in this process together with ``lane``.  ``device``:
    where the writer's kernel runs (default: the current device).  The lane must be free: a second writer of a lane is
    refused.  ``timeout``: seconds a commit waits, retrying, for the learner to free a slot before TimeoutError.

    ``append_vector_step`` has the signature and n_new rule of ``ReplayDataset.append_vector_step``, so a ``ShardActor``
    takes the writer as its sink.  Each stream is reset on the writer's first step (the writer cannot see the learner's
    index).  Steps are packed into page-locked staging; a full slot is committed when the next step would not fit, or on
    ``flush()``."""

    def __init__(self, handle, device=None, lane=None, timeout=30.0):
        own = isinstance(handle, TransitionInbox)
        self.lib = _lib.load()
        if own:
            if lane is None:
                raise ValueError("TransitionWriter(inbox, lane=): an in-process writer names its lane")
            fields = dict(lane=int(lane), lanes=handle.lanes, slots=handle.slots, slot_transitions=handle.T,
                          slot_frames=handle.SF, frame_bytes=handle.F, frame_shape=tuple(handle.replay.frame_shape),
                          streams_per_lane=handle.E, n_gather=handle.replay.n_gather, layout=handle.layout)
        else:
            fields = handle
        self.lane = int(fields["lane"])
        self.T, self.SF, self.F = int(fields["slot_transitions"]), int(fields["slot_frames"]), int(fields["frame_bytes"])
        self.E, self.n_gather = int(fields["streams_per_lane"]), int(fields["n_gather"])
        self.frame_shape = tuple(fields["frame_shape"])
        self.layout = slot_layout(self.T, self.SF, self.F, fields["lanes"], fields["slots"])
        if self.layout != dict(fields["layout"]):
            raise ValueError(f"the inbox's slot layout {fields['layout']} is not this library's {self.layout}")
        self.timeout = float(timeout)
        if own:
            self.device = handle.device
        else:
            self.device = torch.device(device if device is not None else "cuda")
            if self.device.index is None:
                self.device = torch.device("cuda", torch.cuda.current_device())
        w = C.c_void_p()
        with torch.cuda.device(self.device):
            if own:
                _lib.check(self.lib.a0_tw_attach(C.byref(w), handle._h, self.lane), "a0_tw_attach")
                self._inbox = handle                                  # keeps the region alive
            else:
                ipc = (C.c_uint8 * 64).from_buffer_copy(fields["ipc"])
                _lib.check(self.lib.a0_tw_open(C.byref(w), ipc, self.lane, self.F, self.T, self.SF, self.device.index),
                           "a0_tw_open")
        self._h = w
        nbytes = self.layout["slot_bytes"]
        self._host = torch.zeros(nbytes, dtype=torch.uint8).pin_memory()
        self._dev = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        self._status_host = torch.zeros(1, dtype=torch.int64).pin_memory()
        self._status_mapped = _lib.host_map(self._status_host)
        self.packer = SlotPacker(self._host.numpy(), self.layout, self.T, self.SF, self.F)
        self._started = False
        self.committed = 0                                            # slots committed by this writer

    def append_vector_step(self, obs, action, reward, done, obs_next):
        """ReplayDataset.append_vector_step for the writer's E streams.  When the step does not fit the slot, the slot is
        committed first; a TimeoutError from that commit leaves the step untaken (call again)."""
        obs, obs_next = np.asarray(obs, dtype=np.uint8), np.asarray(obs_next, dtype=np.uint8)
        E = obs.shape[0]
        if E != self.E or obs.shape[1:] != (4,) + self.frame_shape or obs_next.shape != obs.shape:
            raise ValueError(f"the lane takes steps of {self.E} streams of [4, {self.frame_shape}] stacks, not {obs.shape}")
        k = stack_delta(obs, obs_next)
        reset = not self._started
        new = [obs_next[e, 4 - k[e]:] for e in range(E) if k[e]]
        parts = ([obs.reshape(4 * E, self.F)] if reset else []) + [x.reshape(-1, self.F) for x in new]
        frames = np.concatenate(parts) if parts else np.zeros((0, self.F), dtype=np.uint8)
        if not self.packer.fits(E, len(frames)):
            self.flush()
            if not self.packer.fits(E, len(frames)):
                raise ValueError(f"a vector step of {E} transitions and {len(frames)} frames does not fit a slot "
                                 f"({self.T} transitions, {self.SF} frames)")
        self.packer.add(reset, np.arange(E, dtype=np.int64), k, np.asarray(action, dtype=np.int64),
                        np.asarray(reward, dtype=np.float64), done, frames)
        self._started = True

    def flush(self):
        """Commits the packed steps (if any) as one slot: one H2D copy, then K9a, then a synchronise.  While every slot
        of the lane waits for the learner, retries every half millisecond; TimeoutError after ``timeout`` seconds (the
        steps stay packed).  Returns the transitions committed."""
        p = self.packer
        if p.n_transitions == 0:
            return 0
        nbytes = p.nbytes()
        deadline = time.monotonic() + self.timeout
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream(self.device)
            self._dev[:nbytes].copy_(self._host[:nbytes], non_blocking=True)
            while True:
                self._status_host.zero_()
                _lib.check(self.lib.a0_tw_commit(self._h, self._dev.data_ptr(), p.n_transitions, p.n_steps, p.n_frames,
                                                 self._status_mapped, _lib.stream_ptr(self.device)), "a0_tw_commit")
                stream.synchronize()
                status = int(self._status_host[0])
                if status == _lib.TX_COMMITTED:
                    break
                if status != _lib.TX_FULL:
                    raise RuntimeError(f"a0_tw_commit: unexpected status {status}")
                if time.monotonic() >= deadline:
                    raise TimeoutError(f"transition inbox lane {self.lane}: every slot still waits for the learner after "
                                       f"{self.timeout} s")
                time.sleep(0.0005)
        n = p.n_transitions
        p.clear()
        self.committed += 1
        return n

    def close(self):
        """Hands the lane back (steps not flushed are dropped)."""
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.a0_tw_close(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
