"""Shard checkpoints merged into shards of another capacity or world size (a0_ckpt_merge, ReplayDataset.load_merged,
Trainer.load across world sizes): every record the target keeps gathers bit-identically to the same record on its
source shard (frames of the n-step window, action, reward as float64, done, boot index through the record map); leaves
are the source leaves and the tree is the oracle's; max_p and the call counter are the maxima over the files; the index
is a0_ix_merge's on the files' host data; ingest continues on carried streams; corrupt or mismatched files raise and
leave the shard as it was (or empty, for a bad blob); a graph captured before a merge replays correctly after it; a
Trainer resumes on one rank from two and on two ranks from one."""
import os
import struct

import numpy as np
import pytest
import torch

from agent0_b200 import _lib
from agent0_b200.config import make_config
from agent0_b200.replay import NORM_DIV, ReplayDataset
from agent0_b200.ring_index import NativeRingIndex
from agent0_b200.synth import fill_shard_synthetic, record_stream
from agent0_b200.trainer import reshard_assignment
from oracle import cpu_path as CP
from oracle import reference_replay as OR
from oracle.sumtree import SumTree

pytestmark = pytest.mark.gpu
E = 4


# ---- fill patterns, as tests/test_gpu_checkpoint.py ----------------------------------------------------------------
def _cfg(kind, size):
    per = kind != "uniform"
    n = 3 if kind in ("nstep", "depth24") else 1
    cfg = make_config("c51", per=per, n_step=n, batch_size=16, replay_size=size, double_q=True, num_envs=E, action_dim=4)
    if kind == "depth24":
        cfg.obs_shape = (4, 4, 4)
    return cfg


def _shard(kind, size, frame_capacity=None):
    return ReplayDataset(_cfg(kind, size), native_nstep=kind in ("nstep", "depth24"), compat_sum=kind == "compat_sum",
                         frame_capacity=frame_capacity)


def _tuples(steps, seed, hw=(84, 84)):
    s = record_stream(E, steps, seed=seed, frame_hw=hw)
    fr, a, r, d = OR.pack_nstep(s["obs"], s["action"], s["reward"], s["done"], 3, 0.99)
    z = CP.lz4()
    return [(z.compress(fr[i].tobytes()), int(a[i]), float(r[i]), bool(d[i])) for i in range(len(a))]


def _fill(rp, kind, seed, amount):
    if kind in ("nstep", "depth24"):
        fill_shard_synthetic(rp, amount, E, seed)
    else:
        tup = _tuples(amount, seed)
        for lo in range(0, len(tup), 256):
            rp.extend(tup[lo:lo + 256])
    if rp.prioritize:
        g = torch.Generator("cuda").manual_seed(seed)
        ids = torch.randint(0, rp.size, (300,), device="cuda", generator=g)
        rp.update_priority(ids, torch.rand(300, device="cuda", generator=g) * 5)
        for _ in range(seed % 3 + 1):
            rp.sample(16, k_batches=2, seed=5)                 # advances the device call counter differently per file
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


def _unchanged(before, rp, what):
    after = _state(rp)
    for k in before:
        v, w = before[k], after[k]
        assert (torch.equal(v, w) if isinstance(v, torch.Tensor) else v == w), (what, k)


# ---- the files' host data -----------------------------------------------------------------------------------------
def _sections(data):
    out, at = {}, 64
    while at < len(data):
        tag, _, ln, _ = struct.unpack_from("<IIQQ", data, at)
        out[tag] = (at + 24, ln)
        at += 24 + ln
    return out


def ck_hash(b):
    """The section hash of a0_ckpt.cu, restated (to build files that pass the hash check)."""
    M = (1 << 64) - 1
    K = 0x9FB21C651E98DF25
    lane = lambda x, w: (((((x ^ w) * K) & M) << 29) | ((((x ^ w) * K) & M) >> 35)) & M
    h = [0x9E3779B97F4A7C15, 0xC2B2AE3D27D4EB4F, 0x165667B19E3779F9, 0x27D4EB2F165667C5]
    n32 = len(b) // 32 * 32
    for row in np.frombuffer(b[:n32], dtype="<u8").reshape(-1, 4).tolist():
        h = [lane(h[i], row[i]) for i in range(4)]
    x = (h[0] ^ (h[1] * 3) ^ (h[2] * 5) ^ (h[3] * 7)) & M
    for c in b[n32:]:
        x = lane(x, c)
    x = lane(x, len(b))
    x ^= x >> 32
    x = (x * 0xD6E8FEB86659FD93) & M
    return x ^ (x >> 32)


def _host(path):
    """(NativeRingIndex, RECORDS bytes, leaves, [(tail id, seq[8])], max_p, call counter) of a checkpoint file."""
    data = open(path, "rb").read()
    N, NF, F, P, n, age = struct.unpack_from("<6q", data, 16)
    s = _sections(data)
    ix = NativeRingIndex(N, NF, n, age)
    ix.deserialize(data[s[1][0]:s[1][0] + s[1][1]])
    rec = data[s[2][0]:s[2][0] + s[2][1]]
    leaves = np.frombuffer(data[s[3][0]:s[3][0] + s[3][1]], dtype="<f4").copy()
    sc = data[s[4][0]:s[4][0] + 32]
    t0 = s[5][0]
    count = struct.unpack_from("<q", data, t0)[0]
    each = 8 + 64 + 8 + 8 * F + 64
    tails = [(struct.unpack_from("<q", data, t0 + 8 + e * each)[0],
              np.frombuffer(data, dtype="<i8", count=8, offset=t0 + 16 + e * each).copy()) for e in range(count)]
    return ix, rec, leaves, tails, struct.unpack_from("<f", sc, 0)[0], struct.unpack_from("<Q", sc, 16)[0]


def _host_merge(rp, paths, streams=None):
    """a0_ix_merge on the files' host data into a fresh index of rp's shape."""
    hs = [_host(p) for p in paths]
    ix = NativeRingIndex(rp.size, rp.index.NF, rp.index.n, rp.index.age_limit)
    out = ix.merge([h[0] for h in hs], [h[1] for h in hs], [h[2] for h in hs], streams, [h[3] for h in hs])
    return ix, out, hs


def _gather(rp, idx, f32=False):
    idx = torch.as_tensor(np.asarray(idx, dtype=np.int64), device="cuda")
    b = rp.gather(idx, normalized=NORM_DIV if f32 else None)
    return b


def _check_records(srcs, dst, out, hs, f32_too=False):
    """Every record the target holds sampleable gathers as its source record; leaves are the source leaves; the tree
    is the oracle's; max_p and the call counter are the maxima over the files."""
    rmap = out["record_map"]
    back = {(int(j), int(s)): int(d) for j, s, d in rmap}
    samp = dst.index.sampleable
    n_checked = 0
    for j, rp in enumerate(srcs):
        rows = rmap[(rmap[:, 0] == j) & (rmap[:, 2] >= 0)]
        rows = rows[samp[rows[:, 2]]]
        for lo in range(0, len(rows), 4096):
            part = rows[lo:lo + 4096]
            a, b = _gather(rp, part[:, 1]), _gather(dst, part[:, 2])
            for f in ("frames", "actions", "rewards", "terminals", "rewards_f32", "terminals_f32"):
                assert torch.equal(getattr(a, f), getattr(b, f)), f
            boot = [x if x < 0 else back.get((j, x), -2) for x in a.boot_indices.cpu().tolist()]
            assert np.array_equal(np.array(boot), b.boot_indices.cpu().numpy())
            if f32_too and lo == 0:
                a32, b32 = _gather(rp, part[:, 1], True), _gather(dst, part[:, 2], True)
                assert torch.equal(a32.obs, b32.obs) and torch.equal(a32.next_obs, b32.next_obs)
            n_checked += len(part)
            st = rp.tree[rp.P + torch.as_tensor(part[:, 1], device="cuda")]
            assert torch.equal(st, dst.tree[dst.P + torch.as_tensor(part[:, 2], device="cuda")])
    assert n_checked == dst.top > 0
    leaves = dst.tree[dst.P:dst.P + dst.size].cpu().numpy()
    assert np.all(leaves[~samp] == 0)
    assert np.array_equal(leaves, out["leaves"])
    ref = SumTree(dst.size)
    ref.build(leaves)
    assert np.array_equal(dst.tree.cpu().numpy().view(np.int32), ref.nodes.view(np.int32))
    assert dst.max_p == max(h[4] for h in hs)
    calls = max(h[5] for h in hs)
    u1 = torch.empty(16, device="cuda")
    u2 = torch.empty(16, device="cuda")
    dst.sample(16, seed=3, u_out=u1)
    dst.sample(16, seed=3, call=calls, u_out=u2)
    assert torch.equal(u1, u2)


CASES = [("nstep", 1, "larger"), ("nstep", 2, "equal"), ("nstep", 3, "smaller"), ("tuples", 2, "larger"),
         ("tuples", 1, "smaller_frames"), ("uniform", 2, "equal"), ("compat_sum", 3, "larger")]


@pytest.mark.parametrize("kind,k,target", CASES)
def test_merged_records_match_their_sources(kind, k, target, tmp_path):
    size = 1024
    amount = {"nstep": 900, "tuples": 180, "uniform": 200, "compat_sum": 150}
    srcs, paths = [], []
    for j in range(k):
        rp = _shard(kind, size)
        _fill(rp, kind, seed=1 + j, amount=amount[kind] * (j + 1) if kind != "nstep" else 600 + 700 * j)
        p = tmp_path / f"s{j}.a0ckpt"
        rp.save(p)
        srcs.append(rp)
        paths.append(p)
    total = sum(rp.index.head_q - rp.index.tail_q for rp in srcs)
    N2, NF2 = {"larger": (4096, None), "equal": (size, None), "smaller": (total // 2, None),
               "smaller_frames": (4096, 3000)}[target]
    dst = _shard(kind, N2, NF2)
    users = dst.load_merged(paths)
    torch.cuda.synchronize()
    assert len(users) == k and dst.beta == srcs[0].beta
    ix, out, hs = _host_merge(dst, paths)
    assert dst.index.serialize() == ix.serialize()
    if target == "larger":
        assert dst.top == sum(rp.top for rp in srcs)
    _check_records(srcs, dst, out, hs, f32_too=(kind == "nstep" and k == 1))
    # ingest continues on the carried streams, with the same content as on the source
    if kind in ("tuples", "uniform", "compat_sum") and k == 1:
        tup = _tuples(20, 77)
        h0, s0 = dst.index.head_fs, srcs[0].index.head_fs
        dst.extend(tup)
        srcs[0].extend(tup)
        # the remapped tails de-duplicate: no more new frames than on the source, the same content
        assert dst.index.head_fs - h0 <= srcs[0].index.head_fs - s0
        m = len(tup)
        a = _gather(srcs[0], (srcs[0].index.head_q - m + np.arange(m)) % srcs[0].size)
        b = _gather(dst, (dst.index.head_q - m + np.arange(m)) % dst.size)
        assert torch.equal(a.frames, b.frames) and torch.equal(a.rewards, b.rewards) and torch.equal(a.actions, b.actions)
    if kind == "nstep" and k == 1:
        m = 64
        st = np.tile(np.arange(E), m // E)
        fr = torch.randint(0, 256, (m, dst.F), dtype=torch.uint8, device="cuda", generator=torch.Generator("cuda").manual_seed(3))
        for rp in (dst, srcs[0]):
            rp.append_steps(st, np.ones(m, np.int64), fr, np.full(m, 2), np.full(m, 0.25), np.zeros(m, bool))
        torch.cuda.synchronize()
        a = _gather(srcs[0], (srcs[0].index.head_q - m + np.arange(m - 3 * E)) % srcs[0].size)
        b = _gather(dst, (dst.index.head_q - m + np.arange(m - 3 * E)) % dst.size)
        assert torch.equal(a.frames, b.frames) and torch.equal(a.rewards, b.rewards)


def test_depth24_target(tmp_path):
    src = _shard("depth24", 1 << 24)
    _fill(src, "depth24", seed=4, amount=40000)
    p = tmp_path / "d.a0ckpt"
    src.save(p)
    dst = _shard("depth24", 1 << 24)
    dst.load_merged([p])
    torch.cuda.synchronize()
    ix, out, hs = _host_merge(dst, [p])
    assert dst.index.serialize() == ix.serialize() and dst.top == src.top
    _check_records([src], dst, out, hs)


def test_bad_files_raise_and_leave_the_shard_untouched(tmp_path):
    kind = "tuples"
    paths = []
    for j in range(3):
        rp = _shard(kind, 512)
        _fill(rp, kind, seed=10 + j, amount=150)
        paths.append(tmp_path / f"g{j}.a0ckpt")
        rp.save(paths[-1])
    good = paths[1].read_bytes()
    secs = _sections(good)
    dst = _shard(kind, 1024)
    _fill(dst, kind, seed=20, amount=60)
    before = _state(dst)

    def flip(at):
        d = bytearray(good)
        d[at] ^= 0x10
        return bytes(d)

    def patch(tag, fn):
        d = bytearray(good)
        off, ln = secs[tag]
        p = bytearray(d[off:off + ln])
        fn(p)
        d[off:off + ln] = p
        struct.pack_into("<Q", d, off - 8, ck_hash(bytes(p)))
        return bytes(d)

    bad = {"section byte": flip(secs[2][0] + 100), "truncated": good[:len(good) // 2],
           "bad table": patch(7, lambda p: struct.pack_into("<q", p, 24 + 8, 3))}
    for name, data in bad.items():
        f = tmp_path / "bad.a0ckpt"
        f.write_bytes(data)
        with pytest.raises(RuntimeError):
            dst.load_merged([paths[0], f, paths[2]])
        _unchanged(before, dst, name)
    with pytest.raises(RuntimeError, match="both become stream"):
        dst.load_merged(paths[:2], [{0: 1}, {2: 1}])
    _unchanged(before, dst, "ids")
    cfg = _cfg(kind, 512)
    cfg.obs_shape = (4, 4, 4)
    other = ReplayDataset(cfg)
    other.extend([(np.zeros(8 * 16, np.uint8).tobytes(), 0, 0.0, False)])
    of = tmp_path / "f16.a0ckpt"
    other.save(of)
    with pytest.raises(RuntimeError, match="F="):
        dst.load_merged([paths[0], of])
    _unchanged(before, dst, "F")
    # a flipped byte inside a blob is caught while the frames are placed: the shard is left empty
    off, ln = secs[8]
    f = tmp_path / "blob.a0ckpt"
    f.write_bytes(flip(off + ln // 2))
    with pytest.raises(RuntimeError, match="reset to empty"):
        dst.load_merged([paths[0], f])
    torch.cuda.synchronize()
    assert dst.top == 0 and dst.index.head_q == 0 and float(dst.tree.abs().max()) == 0.0 and dst.max_p == 1.0
    dst.load_merged(paths)                                              # and it takes good files afterwards
    assert dst.top > 0


def test_graph_captured_before_a_merge_replays_after_it(tmp_path):
    from agent0_b200.hotloop import ReplayTargetLoop
    from tests.test_gpu_hotloop import _outputs
    B, L, A = 16, 2, 4
    src = _shard("nstep", 1024)
    _fill(src, "nstep", seed=4, amount=900)
    path = tmp_path / "s.a0ckpt"
    src.save(path)
    o = _outputs("c51", B * L)
    a = _shard("nstep", 2048)
    _fill(a, "nstep", seed=5, amount=900)
    loop_a = ReplayTargetLoop(a, "c51", B, L, A, o, n_step=3, rng_seed=9)
    loop_a.capture()
    a.load_merged([path])
    b = _shard("nstep", 2048)
    b.load_merged([path])
    loop_b = ReplayTargetLoop(b, "c51", B, L, A, o, n_step=3, rng_seed=9)
    for rp in (a, b):
        rp.push_dynamic()
    loop_a.run()
    loop_b.step()
    torch.cuda.synchronize()
    assert torch.equal(loop_a.idx, loop_b.idx) and torch.equal(loop_a.w, loop_b.w) and torch.equal(loop_a.frames, loop_b.frames)
    assert torch.equal(loop_a.loss, loop_b.loss) and torch.equal(a.tree, b.tree)


def _trainer_cfg():
    cfg = make_config("c51", per=True, n_step=3, batch_size=8, double_q=True, dueling=True, replay_size=512, num_envs=E)
    cfg.learner.learner_steps = 2
    cfg.learner.target_update_freq = 4
    return cfg


def test_trainer_two_ranks_into_one(tmp_path):
    from agent0_b200.dist import adam_eps
    from agent0_b200.trainer import Trainer
    cfg = _trainer_cfg()
    torch.manual_seed(3)
    a = Trainer(cfg, sampler_seed=21)
    a.replay.extend(_tuples(60, 8))
    a.learn()
    a.save(tmp_path)
    os.remove(tmp_path / "replay.a0ckpt")
    shards = []
    for r in range(2):
        rp = _shard("tuples", 512)
        _fill(rp, "tuples", seed=30 + r, amount=50 + 20 * r)
        rp.save(tmp_path / f"replay.rank{r}.a0ckpt")
        shards.append(rp)
    st = torch.load(tmp_path / "learner.pt", weights_only=False)
    for g in st["optimizer"]["param_groups"]:
        g["eps"] = adam_eps(cfg.learner.batch_size, 2)                 # as a 2-rank run saves it
    torch.save(st, tmp_path / "learner.pt")
    b = Trainer(cfg, sampler_seed=21)
    b.load(tmp_path)
    for pa, pb in zip(a.learner.model.parameters(), b.learner.model.parameters()):
        assert torch.equal(pa, pb)
    assert all(g["eps"] == adam_eps(cfg.learner.batch_size, 1) for g in b.learner.optimizer.param_groups)
    assert b.replay.top == sum(rp.top for rp in shards)
    files = [tmp_path / f"replay.rank{r}.a0ckpt" for r in range(2)]
    plan = reshard_assignment(2, 1, [ReplayDataset.checkpoint_info(f)["streams"] for f in files])
    ix, out, hs = _host_merge(b.replay, files, [m for _, m in plan[0]])
    assert b.replay.index.serialize() == ix.serialize()
    _check_records(shards, b.replay, out, hs)
    b.learn()


def test_trainer_one_rank_into_two(tmp_path):
    from agent0_b200.dist import adam_eps
    from agent0_b200.trainer import Trainer
    cfg = _trainer_cfg()
    a = Trainer(cfg, sampler_seed=21)
    a.replay.extend(_tuples(60, 9))
    a.save(tmp_path)
    info = ReplayDataset.checkpoint_info(tmp_path / "replay.a0ckpt")
    assert info["N"] == 512 and info["sampleable"] == a.replay.top and info["streams"] == list(range(E))
    got = []
    for r in range(2):
        t = Trainer(cfg, sampler_seed=21)
        t.load(tmp_path, rank=r, world=2)
        assert all(g["eps"] == adam_eps(cfg.learner.batch_size, 2) for g in t.learner.optimizer.param_groups)
        ids = ReplayDataset.checkpoint_info(tmp_path / "replay.a0ckpt")["streams"]
        t.replay.save(tmp_path / f"out{r}.a0ckpt")
        got.append(set(ReplayDataset.checkpoint_info(tmp_path / f"out{r}.a0ckpt")["streams"]))
        assert t.replay.top > 0
    assert got[0] | got[1] == set(ids) and not (got[0] & got[1])
