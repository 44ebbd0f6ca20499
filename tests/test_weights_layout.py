"""Weight snapshots (agent0_b200/weights.py, K8) without a GPU: the layout hash that publisher and subscribers agree on,
what a publisher refuses, the handle an actor process receives, and the C ABI's argument checks."""
import ctypes as C
import pickle

import pytest
import torch
import torch.nn as nn

from agent0_b200.config import make_config
from agent0_b200.model import DeepQNet
from agent0_b200.weights import WeightPublisher, WeightSubscriber, layout_hash


class _Two(nn.Module):
    def __init__(self, first="a", shape=(3, 4), swap=False):
        super().__init__()
        mods = [(first, nn.Linear(*shape)), ("b", nn.Linear(2, 2))]
        for k, m in (mods[::-1] if swap else mods):
            self.add_module(k, m)


def _net(seed, algo="c51", **kw):
    torch.manual_seed(seed)
    return DeepQNet(make_config(algo, dueling=True, **kw))


def test_layout_hash_is_stable():
    # the same layout gives the same hash whatever the weights, in every process and release (a pinned value)
    assert layout_hash(_net(0)) == layout_hash(_net(1))
    assert layout_hash(_Two()) == 0x4AF7CA33438C3D75


@pytest.mark.parametrize("change", ["name", "shape", "dtype", "stride", "order"])
def test_layout_hash_changes_with_the_layout(change):
    base = _Two()
    other = {"name": lambda: _Two(first="c"), "shape": lambda: _Two(shape=(3, 5)), "dtype": lambda: _Two().double(),
             "stride": _strided,
             "order": lambda: _Two(swap=True)}[change]()
    assert layout_hash(other) != layout_hash(base)


def _strided():
    m = _Two()
    with torch.no_grad():
        m.a.weight = nn.Parameter(m.a.weight.detach().t().contiguous().t())     # same shape, column-major storage
    return m


def test_channels_last_network_has_its_own_layout():
    net = _net(0)
    assert layout_hash(net.to(memory_format=torch.channels_last)) != layout_hash(_net(0))


@pytest.mark.parametrize("kind", ["float64", "int_buffer", "bf16"])
def test_non_fp32_state_is_refused(kind):
    m = _Two()
    if kind == "float64":
        m = m.double()
    elif kind == "bf16":
        m = m.to(torch.bfloat16)
    else:
        m.register_buffer("count", torch.zeros(3, dtype=torch.int64))
    with pytest.raises(TypeError, match="4-byte floating-point"):
        WeightPublisher(m)


def test_handle_pickles_and_a_mismatched_layout_is_refused_before_any_copy():
    net = _net(0)
    handle = dict(ipc=bytes(range(64)), n_words=sum(t.numel() for t in net.state_dict().values()),
                  layout_hash=layout_hash(net), pci_bus_id="0000:1b:00.0")
    back = pickle.loads(pickle.dumps(handle))
    assert back == handle
    with pytest.raises(ValueError, match="not the publisher's"):
        WeightSubscriber(back, _net(0, algo="qr"))
    with pytest.raises(ValueError, match="not the publisher's"):
        WeightSubscriber(back, _net(0).to(memory_format=torch.channels_last))


def test_entry_points_reject_bad_arguments_without_a_gpu():
    from agent0_b200 import _lib
    lib = _lib.load()
    h = C.c_void_p()
    buf = (C.c_uint8 * 64)()
    assert lib.a0_wp_create(None, 16, 1, 0) == -1 and b"NULL" in lib.a0_last_error()
    assert lib.a0_wp_create(C.byref(h), 0, 1, 0) == -1 and b"n_words" in lib.a0_last_error()
    assert lib.a0_wp_create(C.byref(h), 1 << 40, 1, 0) == -1
    assert lib.a0_wp_create(C.byref(h), 16, 1, -1) == -1 and b"device" in lib.a0_last_error()
    assert lib.a0_wp_handle(None, buf) == -1
    assert lib.a0_wp_publish(None, None, None, 1, None) == -1 and b"NULL" in lib.a0_last_error()
    assert lib.a0_ws_open(None, buf, 1, 16, 0) == -1
    assert lib.a0_ws_open(C.byref(h), None, 1, 16, 0) == -1
    assert lib.a0_ws_open(C.byref(h), buf, 1, 0, 0) == -1 and b"n_words" in lib.a0_last_error()
    assert lib.a0_ws_open(C.byref(h), buf, 1, 16, -2) == -1
    assert lib.a0_ws_attach(None, None) == -1 and lib.a0_ws_attach(C.byref(h), None) == -1
    assert lib.a0_ws_fetch(None, None, None, 1, None, None) == -1 and b"NULL" in lib.a0_last_error()
    assert lib.a0_wp_ctl(None) is None
    assert lib.a0_wp_destroy(None) == 0 and lib.a0_ws_close(None) == 0
    assert h.value is None                                   # nothing was created
