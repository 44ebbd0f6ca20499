"""The learner's weights for actors in their own processes: versioned snapshots in device memory (K8, a0_weights.cu).

The reference's actor nodes fetch ``model.state_dict()`` from the trainer node at the start of every ``sample`` call
(agent0/deepq/launch.py:33-36,56-61), and the learner never waits for them.  Here the learner's GPU holds the state in
a region of two snapshot buffers: ``WeightPublisher.publish`` copies the model's state into the next buffer (one
launch, capturable: ``Trainer(publish_weights=True)`` makes it the last node of the step's CUDA graph), and a
``WeightSubscriber`` in any process on the node -- on the same GPU through CUDA IPC, on a peer GPU over NVLink --
pulls the newest complete version into its own model whenever it likes: no host round trip to the learner, no
collective, no waiting for the writer.  A pull that raced two publishes (torn) applies nothing and returns 0.

The layout is ``actor.flat_state(model)``: parameters and buffers in state_dict order, which is what launch.py ships
and what ``broadcast_model`` sends.  Every tensor must be float32 and dense; they are copied in memory order, so the
layout hash covers names, shapes, dtypes and strides (a channels-last model and a contiguous one do not match).
"""
from __future__ import annotations

import ctypes as C
import hashlib

import torch

from . import _lib


def _dense(t):
    """The tensor's elements fill numel() consecutive elements of its storage (any dimension order)."""
    expect = 1
    for stride, size in sorted((st, s) for s, st in zip(t.shape, t.stride()) if s > 1):
        if stride != expect:
            return False
        expect *= size
    return True


def _state_items(model, check=True):
    """(name, tensor) of the state in state_dict order; check: raise for anything but dense float32 tensors."""
    items = [(k, t) for k, t in model.state_dict().items() if torch.is_tensor(t)]
    if not items:
        raise ValueError("the model has no state tensors")
    for k, t in items if check else ():
        if t.dtype != torch.float32:
            raise TypeError(f"weight snapshots carry 4-byte floating-point state only; {k} is {t.dtype}")
        if not _dense(t):
            raise ValueError(f"{k} does not cover its memory densely (shape {tuple(t.shape)}, stride {t.stride()})")
    return items


def layout_hash(model):
    """64-bit hash of the state layout: every tensor's name, shape, dtype and strides, in state_dict order.  The same
    in every process (no Python ``hash``)."""
    desc = ";".join(f"{k}|{tuple(t.shape)}|{t.dtype}|{t.stride()}" for k, t in _state_items(model, check=False))
    return int.from_bytes(hashlib.blake2b(desc.encode(), digest_size=8).digest(), "little")


class _Segments:
    """The device-side segment table of a model's state: u64 addresses and i64 word-count prefix sums."""

    def __init__(self, model, device):
        self.tensors = [t for _, t in _state_items(model)]        # keeps the storages (and the addresses) alive
        for t in self.tensors:
            if t.device != device:
                raise ValueError(f"every state tensor must live on {device}; found one on {t.device}")
        words = [t.numel() for t in self.tensors]
        pre = [0]
        for w in words:
            pre.append(pre[-1] + w)
        self.n_words, self.n_seg = pre[-1], len(words)
        self.ptr = torch.tensor([t.data_ptr() for t in self.tensors], dtype=torch.int64, device=device)
        self.pre = torch.tensor(pre, dtype=torch.int64, device=device)


def _cuda_device(model, device):
    dev = torch.device(device if device is not None else next(iter(model.state_dict().values())).device)
    if dev.type != "cuda":
        raise RuntimeError("weight snapshots live in CUDA device memory (there is no CPU path)")
    return torch.device("cuda", dev.index if dev.index is not None else torch.cuda.current_device())


class WeightPublisher:
    """Publishes ``model``'s state (the learner's online network) as versions 1, 2, ... into a device region that
    subscribers map.  ``publish`` enqueues one kernel on the current stream and can be captured in a CUDA graph."""

    def __init__(self, model, device=None):
        _state_items(model)
        self.lib = _lib.load()
        self.device = _cuda_device(model, device)
        self.model = model
        self.hash = layout_hash(model)
        self.seg = _Segments(model, self.device)
        self.n_words = self.seg.n_words
        h = C.c_void_p()
        _lib.check(self.lib.a0_wp_create(C.byref(h), self.n_words, self.hash, self.device.index), "a0_wp_create")
        self._h = h

    def publish(self):
        """Copies the current state into the next snapshot (stream-ordered after whatever wrote it)."""
        _lib.check(self.lib.a0_wp_publish(self._h, self.seg.ptr.data_ptr(), self.seg.pre.data_ptr(), self.seg.n_seg,
                                          _lib.stream_ptr(self.device)), "a0_wp_publish")

    def handle(self):
        """What an actor process needs to subscribe (picklable): the IPC handle, the word count, the layout hash and
        the PCI bus id of the publisher's GPU."""
        buf = (C.c_uint8 * 64)()
        _lib.check(self.lib.a0_wp_handle(self._h, buf), "a0_wp_handle")
        return dict(ipc=bytes(buf), n_words=self.n_words, layout_hash=self.hash,
                    pci_bus_id=_lib.pci_bus_id(self.device.index))

    def control_words(self):
        """TEST HOOK: the region's control block as a u64[32] device view (magic | format, hash, n_words, latest,
        seq[0], seq[1], ...)."""
        return _lib.device_view(self.lib.a0_wp_ctl(self._h), (32,), "<i8", self.device, owner=self)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.a0_wp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class WeightSubscriber:
    """Pulls the newest complete snapshot of a ``WeightPublisher`` into ``model``'s state tensors (in place).

    ``handle``: ``WeightPublisher.handle()`` from another process (mapped with CUDA IPC; on another GPU of the node
    the reads go over NVLink), or the ``WeightPublisher`` itself in this process.  ``device``: where ``model`` lives
    (default: its tensors' device).  A model whose layout differs from the publisher's is refused before anything is
    copied.  The publisher must outlive its subscribers."""

    def __init__(self, handle, model, device=None):
        own = isinstance(handle, WeightPublisher)
        want_hash, want_words = (handle.hash, handle.n_words) if own else (int(handle["layout_hash"]), int(handle["n_words"]))
        got, words = layout_hash(model), sum(t.numel() for _, t in _state_items(model))
        if got != want_hash or words != want_words:
            raise ValueError(f"the model's state layout (hash {got:016x}, {words} words) is not the "
                             f"publisher's (hash {want_hash:016x}, {want_words} words)")
        self.lib = _lib.load()
        self.device = _cuda_device(model, device)
        self.model = model
        self.seg = _Segments(model, self.device)
        h = C.c_void_p()
        if own:
            if handle.device != self.device:
                raise ValueError("an in-process subscriber shares the publisher's GPU; use handle() from a process on "
                                 "the other GPU")
            _lib.check(self.lib.a0_ws_attach(C.byref(h), handle._h), "a0_ws_attach")
            self._publisher = handle                               # keeps the region alive
        else:
            ipc = (C.c_uint8 * 64).from_buffer_copy(handle["ipc"])
            _lib.check(self.lib.a0_ws_open(C.byref(h), ipc, want_hash, want_words, self.device.index), "a0_ws_open")
        self._h = h
        self.version = 0                                           # last version pull() applied
        self._status_host = torch.zeros(1, dtype=torch.int64).pin_memory()
        self._status_mapped = _lib.host_map(self._status_host)
        self._status_dev = torch.zeros(1, dtype=torch.int64, device=self.device)

    def _fetch(self, status_ptr):
        _lib.check(self.lib.a0_ws_fetch(self._h, self.seg.ptr.data_ptr(), self.seg.pre.data_ptr(), self.seg.n_seg,
                                        status_ptr, _lib.stream_ptr(self.device)), "a0_ws_fetch")

    def pull(self):
        """Applies the newest complete version if it is newer than the last one applied.  Returns that version, or 0
        (nothing published yet, nothing new, or torn by concurrent publishes: the model is unchanged).  Synchronises
        the current stream once."""
        self._status_host.zero_()
        with torch.cuda.device(self.device):
            self._fetch(self._status_mapped)
            torch.cuda.current_stream(self.device).synchronize()
        v = int(self._status_host[0])
        if v:
            self.version = v
        return v

    def pull_async(self):
        """``pull`` without the synchronisation: returns an i64[1] device tensor that receives the status."""
        with torch.cuda.device(self.device):
            self._fetch(self._status_dev.data_ptr())
        return self._status_dev

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.a0_ws_close(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
