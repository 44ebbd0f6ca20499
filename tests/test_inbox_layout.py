"""The transition inbox (agent0_b200/inbox.py, K9) without a GPU: the region layout, the handle an actor process
receives, the writer's packing and the drain's validation of a slot as host code, and the C ABI's argument checks."""
import ctypes as C
import pickle
import subprocess
import sys

import numpy as np
import pytest

from agent0_b200.inbox import LAYOUT_FIELDS, SlotPacker, TransitionWriter, parse_slot, slot_layout
from agent0_b200.ring_index import stack_delta
from agent0_b200.synth import record_stream

F = 84 * 84


@pytest.mark.parametrize("T,SF,frame_bytes,lanes,slots", [(1280, 2624, F, 8, 4), (1, 4, 16, 1, 1), (17, 39, 48, 3, 5),
                                                           (16, 100, 25600, 2, 2)])
def test_layout_is_aligned_and_disjoint(T, SF, frame_bytes, lanes, slots):
    L = slot_layout(T, SF, frame_bytes, lanes, slots)
    sizes = dict(step_count=8 * T, step_reset=T, stream=8 * T, n_new=8 * T, action=8 * T, reward=8 * T, done=T)
    at = 256                                                  # the slot header
    for k in ("step_count", "step_reset", "stream", "n_new", "action", "reward", "done"):
        assert L[k] % 16 == 0 and L[k] >= at, k
        at = L[k] + sizes[k]
    assert L["frames"] % 256 == 0 and L["frames"] >= at
    assert L["slot_bytes"] % 256 == 0 and L["slot_bytes"] >= L["frames"] + SF * frame_bytes
    assert L["ctl_bytes"] == 256 and L["lane_header_bytes"] == 512
    assert L["lane_bytes"] == 512 + slots * L["slot_bytes"]
    assert L["region_bytes"] == 256 + lanes * L["lane_bytes"]
    assert L["scan_meta"] % 256 == 0 and L["scan_meta"] >= 32 * lanes
    assert L["scan_bytes"] == L["scan_meta"] + lanes * slots * L["frames"]


def test_layout_is_the_same_in_another_process():
    args = (1280, 2624, F, 8, 4)
    code = f"from agent0_b200.inbox import slot_layout; print(sorted(slot_layout(*{args}).items()))"
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, check=True,
                         cwd=__file__.rsplit("/tests/", 1)[0]).stdout.strip()
    assert out == str(sorted(slot_layout(*args).items()))
    assert set(slot_layout(*args)) == set(LAYOUT_FIELDS)


def _handle(**over):
    T, SF, lanes, slots = 64, 140, 2, 4
    h = dict(ipc=bytes(range(64)), lane=1, lanes=lanes, slots=slots, slot_transitions=T, slot_frames=SF, frame_bytes=F,
             frame_shape=(84, 84), streams_per_lane=16, n_gather=3, layout=slot_layout(T, SF, F, lanes, slots),
             pci_bus_id="0000:1b:00.0")
    h.update(over)
    return h


def test_handle_pickles_and_a_mismatched_layout_is_refused_before_mapping():
    h = _handle()
    assert pickle.loads(pickle.dumps(h)) == h
    bad = dict(h["layout"], frames=h["layout"]["frames"] + 256)
    with pytest.raises(ValueError, match="slot layout"):
        TransitionWriter(_handle(layout=bad))
    with pytest.raises(ValueError, match="slot layout"):                  # the layout of another slot size
        TransitionWriter(_handle(slot_frames=141))


def _stream(E, steps, seed, hw=(8, 8)):
    return record_stream(E, steps, seed, frame_hw=hw, p_terminal=0.05, p_life_loss=0.05, p_truncated=0.03)


def _pack(s, E, steps, T, SF, Fb, reset_first=True):
    L = slot_layout(T, SF, Fb)
    buf = np.zeros(L["slot_bytes"], dtype=np.uint8)
    p = SlotPacker(buf, L, T, SF, Fb)
    want = []
    for k in range(steps):
        obs, nxt = s["obs"][k], s["obs"][k + 1]
        d = stack_delta(obs, nxt)
        reset = reset_first and k == 0
        parts = ([obs.reshape(4 * E, Fb)] if reset else []) + [nxt[e, 4 - d[e]:].reshape(-1, Fb) for e in range(E)]
        frames = np.concatenate(parts)
        p.add(reset, np.arange(E), d, s["action"][k], s["reward"][k], s["done"][k], frames)
        want.append((reset, d, frames))
    return L, buf, p, want


def test_a_packed_slot_parses_back_to_the_steps_it_was_packed_from():
    E, steps, Fb = 5, 9, 64
    s = _stream(E, steps, 3)
    T, SF = E * steps, 2 * E * steps + 4 * E
    L, buf, p, want = _pack(s, E, steps, T, SF, Fb)
    assert p.nbytes() == L["frames"] + p.n_frames * Fb
    got = parse_slot(buf[:L["frames"]], L, T, SF, E)
    assert len(got) == steps
    frames = buf[L["frames"]:L["frames"] + SF * Fb].reshape(SF, Fb)
    for k, (st, (reset, d, fr)) in enumerate(zip(got, want)):
        assert st.reset == reset
        assert np.array_equal(st.stream, np.arange(E)) and np.array_equal(st.n_new, d)
        assert np.array_equal(st.action, s["action"][k]) and np.array_equal(st.reward, s["reward"][k])
        assert np.array_equal(st.done.astype(bool), s["done"][k])
        assert np.array_equal(frames[st.frame_off:st.frame_off + st.n_frames], fr)
    assert got[-1].frame_off + got[-1].n_frames == p.n_frames


def test_packer_capacity():
    E, Fb = 4, 16
    s = _stream(E, 3, 4, hw=(4, 4))
    L = slot_layout(8, 40, Fb)
    p = SlotPacker(np.zeros(L["slot_bytes"], dtype=np.uint8), L, 8, 40, Fb)
    assert p.fits(E, 20) and not p.fits(9, 0) and not p.fits(E, 41)
    p.add(True, np.arange(E), np.ones(E, np.int64), s["action"][0], s["reward"][0], s["done"][0],
          np.zeros((4 * E + E, Fb), np.uint8))
    assert p.fits(E, 20) and not p.fits(E, 21) and not p.fits(E + 1, 0)
    p.clear()
    assert p.n_transitions == p.n_steps == p.n_frames == 0


def _corrupt(kind, buf, L, E, T, SF):
    i64 = lambda k: buf[L[k]:L[k] + 8 * T].view(np.int64)
    u8 = lambda k: buf[L[k]:L[k] + T]
    hdr = buf[:24].view(np.int64)
    if kind == "no_transitions":
        hdr[0] = 0
    elif kind == "too_many_transitions":
        hdr[0] = T + 1
    elif kind == "no_steps":
        hdr[1] = 0
    elif kind == "more_steps_than_transitions":
        hdr[1] = hdr[0] + 1
    elif kind == "too_many_frames":
        hdr[2] = SF + 1
    elif kind == "negative_frames":
        hdr[2] = -1
    elif kind == "frames_do_not_add_up":
        hdr[2] -= 1
    elif kind == "step_count_zero":
        i64("step_count")[1] = 0
    elif kind == "step_count_over_streams":
        i64("step_count")[0] = E + 1
    elif kind == "steps_do_not_sum":
        hdr[0] -= 1
    elif kind == "reset_flag":
        u8("step_reset")[2] = 2
    elif kind == "stream_negative":
        i64("stream")[3] = -1
    elif kind == "stream_over":
        i64("stream")[3] = E
    elif kind == "n_new_negative":
        i64("n_new")[5] = -1
    elif kind == "n_new_over":
        i64("n_new")[5] = 5
    elif kind == "done_flag":
        u8("done")[6] = 7
    elif kind == "reset_without_frames":
        u8("step_reset")[1] = 1
    else:
        raise AssertionError(kind)


MALFORMED = ["no_transitions", "too_many_transitions", "no_steps", "more_steps_than_transitions", "too_many_frames",
             "negative_frames", "frames_do_not_add_up", "step_count_zero", "step_count_over_streams", "steps_do_not_sum",
             "reset_flag", "stream_negative", "stream_over", "n_new_negative", "n_new_over", "done_flag",
             "reset_without_frames"]


@pytest.mark.parametrize("kind", MALFORMED)
def test_every_malformed_slot_is_rejected(kind):
    E, steps, Fb = 4, 6, 16
    s = _stream(E, steps, 7, hw=(4, 4))
    T, SF = E * steps, 2 * E * steps + 4 * E
    L, buf, p, _ = _pack(s, E, steps, T, SF, Fb)
    parse_slot(buf[:L["frames"]], L, T, SF, E)                          # well formed before
    _corrupt(kind, buf, L, E, T, SF)
    with pytest.raises(RuntimeError, match="lane 3, slot 1 is malformed"):
        parse_slot(buf[:L["frames"]], L, T, SF, E, where="lane 3, slot 1")


def test_entry_points_reject_bad_arguments_without_a_gpu():
    from agent0_b200 import _lib
    lib = _lib.load()
    h = C.c_void_p()
    buf = (C.c_uint8 * 64)()
    out = np.zeros(15, dtype=np.int64)
    assert lib.a0_tx_layout(16, 40, F, 1, 1, None) == -1 and b"NULL" in lib.a0_last_error()
    assert lib.a0_tx_layout(0, 40, F, 1, 1, out.ctypes.data) == -1 and b"slot_transitions" in lib.a0_last_error()
    assert lib.a0_tx_layout(16, 3, F, 1, 1, out.ctypes.data) == -1 and b"slot_frames" in lib.a0_last_error()
    assert lib.a0_tx_layout(16, 40, 24, 1, 1, out.ctypes.data) == -1 and b"frame_bytes" in lib.a0_last_error()
    assert lib.a0_tx_layout(16, 40, F, 0, 1, out.ctypes.data) == -1 and b"lanes" in lib.a0_last_error()
    assert lib.a0_tx_layout(16, 40, F, 1, 65, out.ctypes.data) == -1 and b"slots" in lib.a0_last_error()
    assert lib.a0_tx_create(None, 1, 1, 16, 40, F, 16, 3, 0) == -1 and b"NULL" in lib.a0_last_error()
    assert lib.a0_tx_create(C.byref(h), 0, 1, 16, 40, F, 16, 3, 0) == -1 and b"lanes" in lib.a0_last_error()
    assert lib.a0_tx_create(C.byref(h), 1, 0, 16, 40, F, 16, 3, 0) == -1 and b"slots" in lib.a0_last_error()
    assert lib.a0_tx_create(C.byref(h), 1, 1, 16, 40, 100, 16, 3, 0) == -1 and b"frame_bytes" in lib.a0_last_error()
    assert lib.a0_tx_create(C.byref(h), 1, 1, 16, 40, F, 0, 3, 0) == -1 and b"streams_per_lane" in lib.a0_last_error()
    assert lib.a0_tx_create(C.byref(h), 1, 1, 16, 40, F, 16, 0, 0) == -1 and b"n_gather" in lib.a0_last_error()
    assert lib.a0_tx_create(C.byref(h), 1, 1, 16, 40, F, 16, 3, -1) == -1 and b"device" in lib.a0_last_error()
    assert lib.a0_tx_handle(None, buf) == -1
    assert lib.a0_tx_scan(None, 1, None) == -1 and lib.a0_tx_release(None, None) == -1
    assert lib.a0_tx_unclaim(None, 0) == -1
    assert lib.a0_tx_ctl(None) is None and lib.a0_tx_scan_host(None) is None and lib.a0_tx_slot_frames(None, 0, 0) is None
    assert lib.a0_tw_open(None, buf, 0, F, 16, 40, 0) == -1
    assert lib.a0_tw_open(C.byref(h), None, 0, F, 16, 40, 0) == -1
    assert lib.a0_tw_open(C.byref(h), buf, -1, F, 16, 40, 0) == -1 and b"lane" in lib.a0_last_error()
    assert lib.a0_tw_open(C.byref(h), buf, 0, 17, 16, 40, 0) == -1 and b"frame_bytes" in lib.a0_last_error()
    assert lib.a0_tw_open(C.byref(h), buf, 0, F, 16, 40, -2) == -1 and b"device" in lib.a0_last_error()
    assert lib.a0_tw_attach(None, None, 0) == -1 and lib.a0_tw_attach(C.byref(h), None, 0) == -1
    assert lib.a0_tw_commit(None, None, 1, 1, 0, None, None) == -1 and b"NULL" in lib.a0_last_error()
    assert lib.a0_tx_destroy(None) == 0 and lib.a0_tw_close(None) == 0
    assert h.value is None                                   # nothing was created
