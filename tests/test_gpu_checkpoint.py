"""Shard checkpoints (a0_ckpt_save / a0_ckpt_load, ReplayDataset.save / load, Trainer.save / load): a loaded shard is
bit-identical to the one that was saved and stays so under the same later sequence of ingests, draws with and without
replacement, priority updates and a graph-replayed ReplayTargetLoop step; corrupt or mismatched files raise
RuntimeError, leaving the shard as it was when validation catches them and empty when the frame decode does; a graph
captured before a load replays correctly after it; a Trainer resumes bit for bit."""
import ctypes as C
import os
import struct

import numpy as np
import pytest
import torch

from agent0_b200 import _lib
from agent0_b200.config import make_config
from agent0_b200.replay import ReplayDataset
from agent0_b200.synth import fill_shard_synthetic, record_stream
from oracle import cpu_path as CP
from oracle import reference_replay as OR

pytestmark = pytest.mark.gpu
E = 4


def _cfg(kind):
    per = kind != "uniform"
    n = 3 if kind == "nstep" else 1
    size = {"unwrapped": 4096, "wrapped": 512, "nstep": 1024, "uniform": 1024, "compat_sum": 1024, "depth24": 1 << 24}[kind]
    cfg = make_config("c51", per=per, n_step=n, batch_size=16, replay_size=size, double_q=True, num_envs=E, action_dim=4)
    if kind == "depth24":
        cfg.obs_shape = (4, 4, 4)
    return cfg


def _shard(kind):
    return ReplayDataset(_cfg(kind), native_nstep=kind in ("nstep", "depth24"), compat_sum=kind == "compat_sum")


def _tuples(steps, seed, hw=(84, 84)):
    s = record_stream(E, steps, seed=seed, frame_hw=hw)
    fr, a, r, d = OR.pack_nstep(s["obs"], s["action"], s["reward"], s["done"], 3, 0.99)
    z = CP.lz4()
    return [(z.compress(fr[i].tobytes()), int(a[i]), float(r[i]), bool(d[i])) for i in range(len(a))]


def _fill(rp, kind, seed):
    if kind in ("nstep", "depth24"):
        fill_shard_synthetic(rp, {"nstep": 2600, "depth24": 40000}[kind], E, seed)
    else:
        tup = _tuples({"unwrapped": 200, "wrapped": 400}.get(kind, 300), seed)
        for lo in range(0, len(tup), 256):
            rp.extend(tup[lo:lo + 256])
    if rp.prioritize:
        g = torch.Generator("cuda").manual_seed(seed)
        ids = torch.randint(0, rp.size, (300,), device="cuda", generator=g)
        rp.update_priority(ids, torch.rand(300, device="cuda", generator=g) * 5)
        rp.sample(16, k_batches=2, seed=5)                 # advances the device call counter
    torch.cuda.synchronize()


def _state(rp):
    lib, dev = rp.lib, rp.device
    ix = rp.index
    hfs = ix.head_fs
    lo = max(0, hfs - ix.NF)
    pos = torch.arange(lo, hfs, device=dev) % ix.NF
    live = (torch.arange(ix.tail_q, ix.head_q, device=dev) % rp.size)
    slots = _lib.device_view(lib.a0_rb_ptr(rp.h, _lib.PTR_REC_SLOTS), (rp.size, 8), "<i4", dev, rp._owner)
    info = _lib.device_view(lib.a0_rb_ptr(rp.h, _lib.PTR_REC_INFO), (rp.size, 4), "<i4", dev, rp._owner)
    scal = _lib.device_view(lib.a0_rb_ptr(rp.h, _lib.PTR_MAX_P), (19,), "<f4", dev, rp._owner)
    return dict(index=ix.serialize(), frames=rp.frames[pos].cpu(), slots=slots[live].cpu(), info=info[live].cpu(),
                tree=rp.tree.cpu(), scalars=scal[[0, 16, 17, 18]].cpu(), beta=rp.beta)


def _same(a, b):
    sa, sb = _state(a), _state(b)
    for k in sa:
        v, w = sa[k], sb[k]
        assert (torch.equal(v, w) if isinstance(v, torch.Tensor) else v == w), k


def _drive(rps, kind, steps=3):
    """The same later sequence on every shard; the draws and the trees must agree at every step."""
    for s in range(steps):
        if kind in ("nstep", "depth24"):
            rng = np.random.RandomState(100 + s)
            m = 64
            st = np.tile(np.arange(E), m // E)
            n_new = np.where(rng.rand(m) < 0.05, 4, 1)
            fr = torch.randint(0, 256, (int(n_new.sum()), rps[0].F), dtype=torch.uint8, device="cuda",
                               generator=torch.Generator("cuda").manual_seed(s))
            for rp in rps:
                rp.append_steps(st, n_new, fr, np.full(m, s % 4), np.full(m, 0.5), np.zeros(m, bool))
        else:
            tup = _tuples(20, 500 + s)
            for rp in rps:
                rp.extend(tup)
        outs = []
        for rp in rps:
            b1 = rp.sample(16, k_batches=2, seed=77)                                  # device call counter
            b2 = rp.sample(8, k_batches=2, replacement=False, seed=13) if rp.prioritize else b1
            outs.append((b1, b2))
            if rp.prioritize:
                rp.update_priority(b1.indices, torch.linspace(0.1, 3.0, b1.indices.numel(), device="cuda"))
        torch.cuda.synchronize()
        for (b1, b2) in outs[1:]:
            for x, y in zip(outs[0][0], b1):
                assert x is None or torch.equal(x, y)
            assert torch.equal(outs[0][1].indices, b2.indices) and torch.equal(outs[0][1].weights, b2.weights)
        for rp in rps[1:]:
            assert torch.equal(rp.tree, rps[0].tree)
            assert float(rp.max_p_tensor) == float(rps[0].max_p_tensor)


@pytest.mark.parametrize("kind", ["unwrapped", "wrapped", "nstep", "uniform", "compat_sum", "depth24"])
def test_resume_is_bit_exact(kind, tmp_path):
    src = _shard(kind)
    _fill(src, kind, seed=1)
    if kind == "wrapped":
        assert src.index.tail_q > 0
    path = tmp_path / "shard.a0ckpt"
    src.save(path)
    dst = _shard(kind)
    dst.load(path)
    torch.cuda.synchronize()
    _same(src, dst)
    assert np.array_equal(src.index.sampleable, dst.index.sampleable) and dst.top == src.top > 0
    _drive([src, dst], kind)
    _same(src, dst)


def _sections(data):
    """[(tag, payload offset, length)] of a checkpoint file."""
    out, at = [], 64
    while at < len(data):
        tag, _, ln, _ = struct.unpack_from("<IIQQ", data, at)
        out.append((tag, at + 24, ln))
        at += 24 + ln
    return out


def ck_hash(b):
    """The section hash of a0_ckpt.cu, restated (to build files that pass the hash check)."""
    M = (1 << 64) - 1
    K = 0x9FB21C651E98DF25
    lane = lambda x, w: (((((x ^ w) * K) & M) << 29) | ((((x ^ w) * K) & M) >> 35)) & M
    h = [0x9E3779B97F4A7C15, 0xC2B2AE3D27D4EB4F, 0x165667B19E3779F9, 0x27D4EB2F165667C5]
    n32 = len(b) // 32 * 32
    w = np.frombuffer(b[:n32], dtype="<u8").reshape(-1, 4)
    for row in w.tolist():
        h = [lane(h[i], row[i]) for i in range(4)]
    x = (h[0] ^ (h[1] * 3) ^ (h[2] * 5) ^ (h[3] * 7)) & M
    for c in b[n32:]:
        x = lane(x, c)
    x = lane(x, len(b))
    x ^= x >> 32
    x = (x * 0xD6E8FEB86659FD93) & M
    return x ^ (x >> 32)


def _patch(data, tag, fn):
    """data with section `tag`'s payload replaced by fn(payload) and its hash recomputed."""
    d = bytearray(data)
    for t, off, ln in _sections(data):
        if t == tag:
            p = bytearray(d[off:off + ln])
            fn(p)
            d[off:off + ln] = p
            struct.pack_into("<Q", d, off - 8, ck_hash(bytes(p)))
    return bytes(d)


def test_corrupt_and_mismatched_checkpoints_raise(tmp_path):
    src = _shard("wrapped")
    _fill(src, "wrapped", seed=2)
    good = tmp_path / "good.a0ckpt"
    src.save(good)
    data = good.read_bytes()
    secs = {t: (off, ln) for t, off, ln in _sections(data)}
    assert sorted(secs) == list(range(1, 9))
    dst = _shard("wrapped")
    _fill(dst, "wrapped", seed=3)
    before = _state(dst)

    def flip(at):
        d = bytearray(data)
        d[at] ^= 0x10
        return bytes(d)

    N = src.size
    leaf_off = secs[3][0]
    rec_off = secs[2][0]
    live_pos = src.index.tail_q % N
    bad = {
        "truncated": data[:len(data) // 2],
        "group table byte": flip(secs[7][0] + 24 + 8),
        "leaf byte": flip(leaf_off + 4 * live_pos + 1),
        "magic": b"X" + data[1:],
        "version": data[:8] + struct.pack("<I", 2) + data[12:],
        "slot out of range": _patch(data, 2, lambda p: struct.pack_into("<i", p, 4 * 8 * live_pos, 1 << 30)),
        "NaN leaf": _patch(data, 3, lambda p: struct.pack_into("<f", p, 4 * live_pos, float("nan"))),
    }
    for name, d in bad.items():
        f = tmp_path / "bad.a0ckpt"
        f.write_bytes(d)
        with pytest.raises(RuntimeError):
            dst.load(f)
        after = _state(dst)
        for k in before:
            assert (torch.equal(before[k], after[k]) if isinstance(before[k], torch.Tensor) else before[k] == after[k]), (name, k)
    for other in (_shard("unwrapped"),):                               # another capacity
        with pytest.raises(RuntimeError, match="N="):
            other.load(good)
    cfg = _cfg("wrapped")
    cfg.obs_shape = (4, 4, 4)                                          # another frame size
    with pytest.raises(RuntimeError, match="F="):
        ReplayDataset(cfg).load(good)
    # a flipped byte inside a blob is caught while the frames are decoded: the shard is left empty
    boff, bln = secs[8]
    f = tmp_path / "blob.a0ckpt"
    f.write_bytes(flip(boff + bln // 2))
    with pytest.raises(RuntimeError, match="reset to empty"):
        dst.load(f)
    torch.cuda.synchronize()
    assert dst.top == 0 and dst.index.head_q == 0 and float(dst.tree.abs().max()) == 0.0 and dst.max_p == 1.0
    dst.load(good)                                                     # and it takes a good file afterwards
    _same(src, dst)


def test_graph_captured_before_a_load_replays_after_it(tmp_path):
    from agent0_b200.hotloop import ReplayTargetLoop
    from tests.test_gpu_hotloop import _outputs
    B, L, A = 16, 2, 4
    src = _shard("nstep")
    _fill(src, "nstep", seed=4)
    path = tmp_path / "s.a0ckpt"
    src.save(path)
    o = _outputs("c51", B * L)
    a = _shard("nstep")
    _fill(a, "nstep", seed=5)
    loop_a = ReplayTargetLoop(a, "c51", B, L, A, o, n_step=3, rng_seed=9)
    loop_a.capture()
    a.load(path)
    b = _shard("nstep")
    b.load(path)
    loop_b = ReplayTargetLoop(b, "c51", B, L, A, o, n_step=3, rng_seed=9)
    for rp in (a, b):
        rp.push_dynamic()
    loop_a.run()
    loop_b.step()
    torch.cuda.synchronize()
    assert torch.equal(loop_a.idx, loop_b.idx) and torch.equal(loop_a.w, loop_b.w) and torch.equal(loop_a.frames, loop_b.frames)
    assert torch.equal(loop_a.loss, loop_b.loss) and torch.equal(a.tree, b.tree)


@pytest.mark.parametrize("graph", [False, True])
def test_trainer_resumes_bit_for_bit(graph, tmp_path):
    from agent0_b200.trainer import Trainer
    det = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    try:
        cfg = make_config("c51", per=True, n_step=3, batch_size=8, double_q=True, dueling=True, replay_size=512, num_envs=E)
        cfg.learner.learner_steps = 2
        cfg.learner.target_update_freq = 4
        tup = _tuples(60, 8)
        torch.manual_seed(3)
        a = Trainer(cfg, graph=graph, sampler_seed=21)
        a.replay.extend(tup)
        for _ in range(3):
            a.learn()
        a.save(tmp_path)
        assert sorted(os.listdir(tmp_path)) == ["learner.pt", "replay.a0ckpt"]
        torch.manual_seed(99)
        b = Trainer(cfg, graph=graph, sampler_seed=21)
        b.load(tmp_path)
        for _ in range(2):
            oa, ob = a.learn(), b.learn()
            torch.cuda.synchronize()
            for (qa, _), (qb, _) in zip(oa, ob):
                assert torch.equal(qa, qb)
        for pa, pb in zip(a.learner.model.parameters(), b.learner.model.parameters()):
            assert torch.equal(pa, pb)
        assert torch.equal(a.replay.tree, b.replay.tree) and a.learner.update_steps == b.learner.update_steps
    finally:
        torch.backends.cudnn.deterministic = det
