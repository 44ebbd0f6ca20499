"""The C-ABI library builds for sm_100a, loads without a GPU, and exports every symbol that
include/agent0_b200.h declares (no compute calls here)."""
import ctypes
import os
import re

from tests.conftest import ROOT


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "agent0_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(a0_[a-z0-9_]+)\s*\(", text)))


def test_library_builds_and_exports_every_declared_symbol():
    from agent0_b200 import build
    lib_path = build.build()
    assert os.path.exists(lib_path)
    lib = ctypes.CDLL(lib_path)
    names = _declared_symbols()
    assert len(names) >= 17
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/agent0_b200.h but not exported"


def test_ctypes_binding_covers_the_header():
    from agent0_b200 import _lib
    assert sorted(_lib.SIGNATURES) == _declared_symbols()
    lib = _lib.load()
    assert lib.a0_version() >= 100
    assert _lib.A0_REC_META_I32 == 14 and _lib.A0_SLOTS == 8


def test_argument_errors_do_not_need_a_gpu():
    from agent0_b200 import _lib
    lib = _lib.load()
    assert lib.a0_rb_reset(None, None) == -1
    assert b"NULL" in lib.a0_last_error()
    assert lib.a0_pt_sample(None, None, 4, 2, 1.0, 0.4, 0.0, 0, None, None, None, None) == -1
    # entry points added for the overlapped sampler/gather pair, the result report and the one-launch ingest
    assert lib.a0_rb_sample_gather(None, None, 1, -1, 4, 2, 1.0, 0.4, 0.0, 0, None, None, None, 3, 0.99, None, None, None, None,
                                   None, None, None, None) == -1
    assert b"handle is NULL" in lib.a0_last_error()
    assert lib.a0_pt_update_report(None, None, None, 4, 0.5, 0.01, None, None, None) == -1
    assert lib.a0_host_map(None, None) == -1 and b"NULL" in lib.a0_last_error()
    assert lib.a0_rb_ingest_steps_dyn(None, None, None, None, None, 0, None, None, None, 0, 0.5, 0.4, 0, None) == -1
    assert lib.a0_rb_gather_bf16(None, None, 4, 3, 0.99, None, None, 0, None, None, None, None, None, None, None) == -1
    for opt, bad in ((6, 9), (3, 0), (2, 5)):
        assert lib.a0_set_option(opt, bad) == -1
    for opt, ok in ((4, 1), (5, 1), (6, 4), (7, 0), (8, 1), (14, 1)):
        assert lib.a0_set_option(opt, ok) == 0
    assert lib.a0_set_option(99, 0) == -1 and b"unknown option" in lib.a0_last_error()


def test_sass_uses_tma_bulk_copies():
    import subprocess
    from agent0_b200 import build
    out = subprocess.run(["cuobjdump", "-sass", build.build()], capture_output=True, text=True).stdout
    assert "UBLKCP" in out and "SYNCS" in out       # cp.async.bulk + mbarrier in the K3 gather
    assert "sm_100a" in subprocess.run(["cuobjdump", "-lelf", build.build()], capture_output=True, text=True).stdout


def test_pyingest_helper_unpacks_the_reference_tuples():
    """csrc/a0_pyingest.c (host glue of ReplayDataset.extend, CPython API): pointers, lengths and the three scalar
    columns of a list of reference tuples -- bytes, bytearray and ndarray blobs, numpy and Python scalars -- and a
    TypeError for a malformed entry."""
    import ctypes as C

    import numpy as np

    from agent0_b200 import _lib, build
    build.build_pyingest()
    h = _lib.pyingest()
    assert h is not None
    rng = np.random.RandomState(0)
    ent = []
    for i in range(50):
        blob = rng.randint(0, 256, rng.randint(1, 300), dtype=np.uint8)
        ent.append(((blob.tobytes(), bytearray(blob.tobytes()), blob)[i % 3], (np.int64(i % 5), i % 5)[i % 2], (np.float64(i) / 7, i / 7)[i % 2],
                    (np.bool_(i % 4 == 0), i % 4 == 0)[i % 2]))
    m = len(ent)
    ptrs = np.zeros(m, np.uint64); lens = np.zeros(m, np.int64); a = np.zeros(m, np.int64); r = np.zeros(m); d = np.zeros(m, np.uint8)
    views = np.zeros(m * int(h.a0_py_buffer_size()), np.uint8)
    assert h.a0_py_unpack(ent, m, ptrs.ctypes.data, lens.ctypes.data, a.ctypes.data, r.ctypes.data, d.ctypes.data, views.ctypes.data) == m
    try:
        for i, (blob, ai, ri, di) in enumerate(ent):
            assert C.string_at(int(ptrs[i]), int(lens[i])) == bytes(blob)
            assert a[i] == int(ai) and r[i] == float(ri) and d[i] == int(bool(di))
    finally:
        h.a0_py_release(m, views.ctypes.data)
    import pytest
    with pytest.raises(TypeError, match="entry 1 is not"):
        h.a0_py_unpack([ent[0], (b"x", 1, 2.0)], 2, ptrs.ctypes.data, lens.ctypes.data, a.ctypes.data, r.ctypes.data, d.ctypes.data, views.ctypes.data)
    with pytest.raises(TypeError):
        h.a0_py_unpack([(b"x", "left", 2.0, False)], 1, ptrs.ctypes.data, lens.ctypes.data, a.ctypes.data, r.ctypes.data, d.ctypes.data, views.ctypes.data)
