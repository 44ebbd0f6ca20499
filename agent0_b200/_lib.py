"""ctypes binding of libagent0_b200.so (the C ABI declared in include/agent0_b200.h).

There is no CPU fallback: if the shared object is missing or a call fails, this raises.
"""
import ctypes as C
import os

import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("A0_LIB") or os.path.join(_PKG, "libagent0_b200.so")   # A0_LIB: the -DA0_TRACE build (tools/trace_step.py)

A0_SLOTS = 8
A0_REC_META_I32 = 14
A0_MAX_NSTEP = 16
A0_MAX_ACTIONS = 32
A0_MAX_QUANTILES = 256
PTR_FRAMES, PTR_REC_SLOTS, PTR_REC_INFO, PTR_TREE, PTR_MAX_P = range(5)
OPT_PDL = 1          # include/agent0_b200.h: A0_OPT_PDL (mask of kernel classes launched programmatically; bit 0 = K4)
K2B_PLAN_MAX = 1024  # include/agent0_b200.h: A0_K2B_PLAN_MAX (largest index count of a0_pt_update_plan / _apply)
K2B_PLAN_BYTES = 90176  # A0_K2B_PLAN_BYTES (the plan buffer)
C51_EARLY = 1        # include/agent0_b200.h: A0_C51_EARLY (a0_loss_c51_linked: batch-side work before the wait)
TX_COMMITTED, TX_FULL = 1, 2   # include/agent0_b200.h: A0_TX_COMMITTED / A0_TX_FULL (a0_tw_commit's status)


def lz4_stride(frame_bytes):
    """include/agent0_b200.h: A0_LZ4_STRIDE -- bytes between the groups of a0_lz4_encode's output."""
    n = 8 * int(frame_bytes)
    return (n + n // 255 + 20 + 15) // 16 * 16

_vp, _i32, _i64, _f32, _f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_double


class LossCommon(C.Structure):
    """a0_loss_common_t"""
    _fields_ = [("B", _i32), ("A", _i32), ("action", _vp), ("reward", _vp), ("done", _vp),
                ("weight", _vp), ("gamma_n", _f32), ("alpha", _f32), ("eps", _f32),
                ("loss", _vp), ("prio", _vp), ("max_p", _vp)]


class Plan(C.Structure):
    """a0_plan_t"""
    _fields_ = [("m", _i32), ("n_new", _i32), ("n_marks", _i32), ("new_frame_pos", C.POINTER(_i32)),
                ("rec_meta", C.POINTER(_i32)), ("marks", C.POINTER(_i32))]


class Merge(C.Structure):
    """a0_merge_t"""
    _fields_ = [("n_place", _i64), ("place", C.POINTER(_i64)), ("n_rec", _i64), ("record_map", C.POINTER(_i64)),
                ("n_tail", _i64), ("tails", C.POINTER(_i64)), ("stride_hint", _i64)]


IX_HEAD_Q, IX_TAIL_Q, IX_HEAD_FS, IX_TOP, IX_REC_CAPACITY, IX_FRAME_CAPACITY, IX_NSTEP, IX_AGE_LIMIT, \
    IX_MAX_CHUNK, IX_STATE_WORDS = range(10)
INGEST_FRAMES_ON_DEVICE, INGEST_FRAMES_PINNED, INGEST_COPY_STREAM = 1, 2, 4

# name -> (restype, argtypes): every symbol include/agent0_b200.h declares
SIGNATURES = {
    "a0_version": (_i32, []),
    "a0_last_error": (C.c_char_p, []),
    "a0_set_option": (_i32, [_i32, _i64]),
    "a0_get_option": (_i32, [_i32, C.POINTER(C.c_int64)]),
    "a0_capture_node": (_i32, [_vp, C.POINTER(_vp)]),
    "a0_capture_join": (_i32, [_vp, _vp]),
    "a0_graph_edges": (_i32, [_vp, _vp, _vp, _vp, _vp, _i64, C.POINTER(_i64)]),
    "a0_rb_create": (_i32, [C.POINTER(_vp), _i64, _i64, _i32, _i32]),
    "a0_rb_destroy": (_i32, [_vp]),
    "a0_rb_reset": (_i32, [_vp, _vp]),
    "a0_rb_ptr": (_vp, [_vp, _i32]),
    "a0_rb_tree_leaves": (_i64, [_vp]),
    "a0_ix_create": (_i32, [C.POINTER(_vp), _i64, _i64, _i32, _i64]),
    "a0_ix_destroy": (_i32, [_vp]),
    "a0_ix_state": (_i32, [_vp, _vp]),
    "a0_ix_sampleable": (_vp, [_vp]),
    "a0_ix_set_stack": (_i32, [_vp, _i64, _vp]),
    "a0_ix_get_stack": (_i32, [_vp, _i64, _vp]),
    "a0_ix_resolve_shift": (_i32, [_vp, _vp, _vp, _i32, _vp]),
    "a0_ix_plan": (_i32, [_vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp, C.POINTER(Plan)]),
    "a0_dd_create": (_i32, [C.POINTER(_vp), _i32]),
    "a0_dd_destroy": (_i32, [_vp]),
    "a0_dd_resolve": (_i32, [_vp, _vp, _vp, _vp, _i32, _vp, _vp, C.POINTER(_i32)]),
    "a0_ex_create": (_i32, [C.POINTER(_vp), _vp, _vp]),
    "a0_ex_destroy": (_i32, [_vp]),
    "a0_ex_extend": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _f32, _vp]),
    "a0_ex_extend_v": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _f32, _vp]),
    "a0_ex_decode": (_i32, [_vp, _vp, _vp, _i32, _vp, _vp, _vp]),
    "a0_ex_resolve": (_i32, [_vp, _vp, _vp, _i32, _vp, _vp, C.POINTER(_i32)]),
    "a0_ex_last_timing": (_i32, [_vp, _vp]),
    "a0_lz4_encode": (_i32, [_vp, _i32, _i32, _vp, _vp, _vp, _vp]),
    "a0_ix_serialize": (_i32, [_vp, _vp, _i64, C.POINTER(_i64)]),
    "a0_ix_deserialize": (_i32, [_vp, _vp, _i64]),
    "a0_ckpt_save": (_i32, [_vp, _vp, _vp, C.c_char_p, _vp, _i64, _vp]),
    "a0_ckpt_load": (_i32, [_vp, _vp, _vp, C.c_char_p, _vp, _i64, C.POINTER(_i64), _vp]),
    "a0_ckpt_last_timing": (_i32, [_vp]),
    "a0_ix_merge": (_i32, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(Merge)]),
    "a0_ckpt_info": (_i32, [C.c_char_p, _vp, _vp, _i64]),
    "a0_ckpt_merge": (_i32, [_vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _i64, _vp, _vp]),
    "a0_rb_ingest_plan": (_i32, [_vp, C.POINTER(Plan), _vp, _vp, _i32, _f32, _vp]),
    "a0_rb_ingest_steps": (_i32, [_vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _i32, _f32, _vp]),
    "a0_rb_ingest_steps_dyn": (_i32, [_vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _i32, _f32, _f32, _i32, _vp]),
    "a0_rb_append": (_i32, [_vp, _vp, _vp, _i32, _vp, _i32, _vp]),
    "a0_pt_mark": (_i32, [_vp, _vp, _i32, _f32, _vp]),
    "a0_pt_update": (_i32, [_vp, _vp, _vp, _i32, _f32, _f32, _vp]),
    "a0_pt_update_report": (_i32, [_vp, _vp, _vp, _i32, _f32, _f32, _vp, _vp, _vp]),
    "a0_pt_update_overlapped": (_i32, [_vp, _vp, _vp, _i32, _f32, _f32, _vp, _vp, _vp]),
    "a0_pt_update_plan": (_i32, [_vp, _vp, _i32, _vp, _vp]),
    "a0_pt_update_apply": (_i32, [_vp, _vp, _vp, _i32, _f32, _f32, _vp, _vp, _vp, _vp]),
    "a0_host_map": (_i32, [_vp, C.POINTER(_vp)]),
    "a0_pt_set": (_i32, [_vp, _vp, _vp, _i32, _vp]),
    "a0_rb_set_dynamic": (_i32, [_vp, _f32, _f32, _f32, _vp]),
    "a0_pt_sample": (_i32, [_vp, _vp, _i32, _i32, _f32, _f32, _f32, _i32, _vp, _vp, _vp, _vp]),
    "a0_pt_sample_rng": (_i32, [_vp, C.c_uint64, _i64, _i32, _i32, _f32, _f32, _f32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "a0_pt_rng_seek": (_i32, [_vp, C.c_uint64, _vp]),
    "a0_pt_sample_unique": (_i32, [_vp, C.c_uint64, _i64, _i32, _i32, _f32, _f32, _f32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "a0_rb_gather": (_i32, [_vp, _vp, _i32, _i32, _f64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp]),
    "a0_rb_sample_gather": (_i32, [_vp, _vp, C.c_uint64, _i64, _i32, _i32, _f32, _f32, _f32, _i32, _vp, _vp, _vp, _i32, _f64,
                                   _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "a0_rb_sample_mail": (_i32, [_vp, _vp, C.c_uint64, _i64, _i32, _i32, _f32, _f32, _f32, _i32, _vp, _vp, _vp, _vp]),
    "a0_rb_gather_mail": (_i32, [_vp, _i32, _i32, _i32, _i32, _f64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "a0_rb_gather_unpaired": (_i32, [_vp, _i32, _vp, _vp]),
    "a0_rb_check_fault": (_i32, [_vp]),
    "a0_rb_gather_f32": (_i32, [_vp, _vp, _i32, _i32, _f64, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "a0_rb_gather_bf16": (_i32, [_vp, _vp, _i32, _i32, _f64, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "a0_loss_dqn": (_i32, [C.POINTER(LossCommon), _vp, _vp, _vp, _vp, _vp]),
    "a0_loss_mdqn": (_i32, [C.POINTER(LossCommon), _vp, _vp, _vp, _f32, _f32, _vp, _vp]),
    "a0_loss_c51": (_i32, [C.POINTER(LossCommon), _vp, _vp, _vp, _vp, _i32, _f32, _f32, _vp, _vp, _vp]),
    "a0_loss_c51_linked": (_i32, [C.POINTER(LossCommon), _vp, _vp, _vp, _vp, _i32, _f32, _f32, _vp, _vp, _i32, _vp]),
    "a0_c51_div_check": (_i32, [_f32, _f32, _i32, _vp, _vp]),
    "a0_loss_quantile": (_i32, [C.POINTER(LossCommon), _i32, _vp, _vp, _vp, _vp, _i32, _i32, _vp,
                                _vp, _vp, _vp, _vp, _vp]),
    "a0_act_epsilon_greedy": (_i32, [_vp, _i32, _i32, _f64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "a0_u8_to_f32": (_i32, [_vp, _vp, _i64, _i32, _vp]),
    "a0_wp_create": (_i32, [C.POINTER(_vp), _i64, C.c_uint64, _i32]),
    "a0_wp_destroy": (_i32, [_vp]),
    "a0_wp_handle": (_i32, [_vp, _vp]),
    "a0_wp_ctl": (_vp, [_vp]),
    "a0_wp_publish": (_i32, [_vp, _vp, _vp, _i32, _vp]),
    "a0_ws_open": (_i32, [C.POINTER(_vp), _vp, C.c_uint64, _i64, _i32]),
    "a0_ws_attach": (_i32, [C.POINTER(_vp), _vp]),
    "a0_ws_fetch": (_i32, [_vp, _vp, _vp, _i32, _vp, _vp]),
    "a0_ws_close": (_i32, [_vp]),
    "a0_tx_layout": (_i32, [_i64, _i64, _i64, _i32, _i32, _vp]),
    "a0_tx_create": (_i32, [C.POINTER(_vp), _i32, _i32, _i64, _i64, _i64, _i32, _i32, _i32]),
    "a0_tx_destroy": (_i32, [_vp]),
    "a0_tx_handle": (_i32, [_vp, _vp]),
    "a0_tx_scan": (_i32, [_vp, _i32, _vp]),
    "a0_tx_scan_host": (_vp, [_vp]),
    "a0_tx_slot_frames": (_vp, [_vp, _i32, _i32]),
    "a0_tx_release": (_i32, [_vp, _vp]),
    "a0_tx_unclaim": (_i32, [_vp, _i32]),
    "a0_tx_ctl": (_vp, [_vp]),
    "a0_tw_open": (_i32, [C.POINTER(_vp), _vp, _i32, _i64, _i64, _i64, _i32]),
    "a0_tw_attach": (_i32, [C.POINTER(_vp), _vp, _i32]),
    "a0_tw_commit": (_i32, [_vp, _vp, _i64, _i64, _i64, _vp, _vp]),
    "a0_tw_close": (_i32, [_vp]),
}

_lib = None


def load():
    """Load the shared object once; raise loudly if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m agent0_b200.build` "
            "(agent0_b200 has no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


_pyingest = False


def pyingest():
    """The CPython-API marshalling helper (csrc/a0_pyingest.c -> _a0_pyingest.so, loaded with PyDLL), or None when
    it has not been built: ``ReplayDataset.extend`` then unpacks the tuples in Python (same C ABI call after that)."""
    global _pyingest
    if _pyingest is False:
        path = os.path.join(_PKG, "_a0_pyingest.so")
        _pyingest = None
        if os.path.exists(path):
            try:
                h = C.PyDLL(path)
                h.a0_py_unpack.restype = _i64
                h.a0_py_unpack.argtypes = [C.py_object, _i64, _vp, _vp, _vp, _vp, _vp, _vp]
                h.a0_py_release.restype = None
                h.a0_py_release.argtypes = [_i64, _vp]
                h.a0_py_buffer_size.restype = _i64
                _pyingest = h
            except OSError:
                _pyingest = None
    return _pyingest


def check(rc, what):
    if rc != 0:
        msg = load().a0_last_error().decode(errors="replace")
        raise RuntimeError(f"{what} failed (code {rc}): {msg}")


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def stream_ptr(device=None):
    """cudaStream_t of torch's current stream on `device` (inside torch.cuda.graph: the capture stream)."""
    if _raw_stream is not None:
        if device is None:
            idx = torch.cuda.current_device()
        elif isinstance(device, int):
            idx = device
        else:
            idx = device.index if device.index is not None else torch.cuda.current_device()
        return _raw_stream(idx)
    return torch.cuda.current_stream(device).cuda_stream


def ptr(t, dtype=None):
    """Raw device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("agent0_b200 kernels need CUDA tensors (there is no CPU path)")
    if dtype is not None and t.dtype != dtype:
        raise TypeError(f"expected {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError("tensor must be contiguous")
    return t.data_ptr()


def pci_bus_id(index):
    """PCI bus id (domain:bus:device.function) of CUDA device ``index``: names the GPU of a region in the handle an
    actor process receives."""
    p = torch.cuda.get_device_properties(index)
    return f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"


def host_map(t):
    """Device-visible address of a pinned CPU tensor (a0_host_map), for kernels that write results
    straight into host memory."""
    if t.is_cuda or not t.is_pinned():
        raise ValueError("host_map needs a pinned CPU tensor")
    out = _vp()
    check(load().a0_host_map(t.data_ptr(), C.byref(out)), "a0_host_map")
    return out.value


class HandleOwner:
    """Owns an a0_replay_t: destroyed when the last reference goes -- the ReplayDataset's and those of
    the tensors that view the handle's device memory."""

    def __init__(self, lib, handle):
        self.lib, self.handle = lib, handle

    def __del__(self):
        try:
            if self.handle is not None and self.handle.value:
                self.lib.a0_rb_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class _DevView:
    """Zero-copy torch view of handle-owned device memory via __cuda_array_interface__.  torch keeps the
    exporting object alive for as long as the tensor's storage lives, and the object keeps ``owner``."""

    def __init__(self, address, shape, typestr, owner=None):
        self.owner = owner
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr,
                                         "data": (int(address), False), "version": 2}


def device_view(address, shape, typestr, device, owner=None):
    return torch.as_tensor(_DevView(address, shape, typestr, owner), device=device)
