"""Every kernel that moves frames, against its reference, at frame sizes from 16 B to the C ABI's limit of 25 600 B
(tests/frame_cases.py: sizes whose 16-byte vector count is or is not a multiple of 32, the last u16-table and first
u32-table groups of K7, a 64x64 RGB frame, the limit itself).  K1 + K3 (variants 0-3 and the converting gathers) on
native ingest against the oracle's actor packer; the mailbox gather and the gather waves against the single-launch
gather; K6a (both forms) against oracle/lz4_block.py; K6b / K6c through extend against the host deduper; K7 against
encode_greedy and the frame hash restated; the checkpoint round trip; shards of different F in one process; the limit.
Every comparison is bit for bit."""
import ctypes as C
import threading
import time

import numpy as np
import pytest
import torch

from agent0_b200 import _lib
from agent0_b200.config import make_config
from agent0_b200.replay import ReplayDataset
from agent0_b200.ring_index import NativeContentDeduper, NativeRingIndex, RingIndex
from agent0_b200.synth import fill_shard_synthetic, record_stream
from oracle import cpu_path as CP
from oracle import lz4_block as LZ
from oracle import reference_replay as OR
from oracle.lz4_encode import encode_greedy
from tests.frame_cases import IDS, SHAPES, far_blocks, frame_bytes, frame_hash, hw2
from tests.test_gpu_checkpoint import E as CK_E
from tests.test_gpu_checkpoint import _drive, _state
from tests.test_gpu_edges import _stream
from tests.test_gpu_extend import _random_sequences, check_malformed_blocks, k6_kernel  # noqa: F401 (fixture)
from tests.test_gpu_hotloop import A as LOOP_A
from tests.test_gpu_hotloop import _outputs
from tests.test_gpu_lz4_encode import _groups, encode

pytestmark = pytest.mark.gpu
by_size = dict(zip(IDS, SHAPES))


def _np(t):
    return t.detach().cpu().numpy()


def _shard(shape, N, NF, n=1, native=True, algo="dqn", E=4, B=8, age_limit=None):
    """A shard with an explicit small frame ring: the default NF = 1.0625 N + 65 536 would be 1.7 GB at 25 600 B."""
    cfg = make_config(algo, per=True, n_step=n, batch_size=B, replay_size=N, num_envs=E, double_q=True, dueling=True,
                      action_dim=LOOP_A)
    cfg.obs_shape = (4,) + tuple(shape)
    return ReplayDataset(cfg, native_nstep=native, frame_capacity=NF, age_limit=age_limit)


# ---------------------------------------------------------------------------------------------------------- K1 + K3
@pytest.mark.parametrize("n", [1, 3, 6])                  # 6: above 4 the speculative window fetch is off
@pytest.mark.parametrize("shape", SHAPES, ids=IDS)
def test_native_ingest_and_every_gather(shape, n):
    """Ragged multi-stream native ingest (static screens, whole new stacks, dones) until both the record ring and the
    frame ring wrap; host-fed pageable (n = 1), host-fed pinned (n = 3) and device-resident (n = 6) frames.  The live
    records are the ones the specification of the index (agent0_b200.ring_index.RingIndex, fed the same steps) holds
    sampleable, and every one of them gathers to the reference entry through K3 variants 0-3; the f32 gathers
    (/255 correctly rounded, * fl(1/255), .float()) and the bf16 gather equal torch's conversions of the u8 stacks."""
    F = frame_bytes(shape)
    E = {1: 3, 3: 4, 6: 5}[n]
    T, N, NF, age = 60, 96, 200, 25
    obs, n_new, act, rew, done = _stream(E, T, shape, seed=F + n, p_new4=0.15, p_static=0.2)
    rp = _shard(shape, N, NF, n=n, E=E, age_limit=age)
    rp.gamma = 0.97
    spec = RingIndex(N, NF, n, age)
    z = np.zeros(0, np.int64)
    spec.plan(z, np.zeros((0, 8), np.int64), np.arange(4 * E), z, z.astype(np.float64), z.astype(bool))
    last4 = {e: np.arange(4 * e, 4 * e + 4, dtype=np.int64) for e in range(E)}
    rp.reset_streams(np.arange(E), obs[0])
    rng = np.random.RandomState(n)
    hist = {e: [] for e in range(E)}         # per stream: ring positions of its records, in step order
    owner = {}                               # ring position -> (stream, step) of the record it holds
    step_of = np.zeros(E, dtype=np.int64)
    keep, q = [], 0
    while step_of.min() < T:
        es = np.flatnonzero((rng.rand(E) < 0.7) & (step_of < T))
        if len(es) == 0:
            continue
        ks = step_of[es]
        k_new = np.array([n_new[k][e] for e, k in zip(es, ks)], dtype=np.int64)
        new = [obs[k + 1][e, 4 - n_new[k][e]:] for e, k in zip(es, ks) if n_new[k][e]]
        new = np.concatenate(new) if new else np.zeros((0,) + tuple(shape), np.uint8)
        if n == 3:
            new = torch.from_numpy(new).pin_memory()
            keep.append(new)                 # pinned_stable: untouched until the stream has passed
        elif n == 6:
            new = torch.from_numpy(new).cuda()
        a, r, d = [np.array([x[k][e] for e, k in zip(es, ks)]) for x in (act, rew, done)]
        rp.append_steps(es, k_new, new, a, r, d, pinned_stable=n == 3)
        fs8 = spec.resolve_shift(es, k_new, last4)
        spec.plan(es, fs8, np.arange(int(k_new.sum())), a, r, d)
        for e in es:
            owner[q % N] = (e, len(hist[e]))
            hist[e].append(q % N)
            q += 1
        step_of[es] += 1
    torch.cuda.synchronize()
    keep.clear()
    assert q == E * T > N and rp.index.head_fs > NF                # both rings wrapped
    live = np.flatnonzero(_np(rp.priority.leaves()) > 0)
    assert np.array_equal(live, np.flatnonzero(spec.sampleable)) and len(live) == rp.top == spec.top > 10
    fr_ref, a_ref, r_ref, d_ref = OR.pack_nstep(obs, act, rew, done, n, 0.97)
    ref = np.array([(owner[p][1] + n - 1) * E + owner[p][0] for p in live])
    boot_ref = np.array([hist[e][j + n] if j + n < len(hist[e]) else -1 for e, j in (owner[p] for p in live)])
    idx = torch.as_tensor(live, device="cuda")
    for variant in (0, 1, 2, 3):
        rp.gather_variant = variant
        b = rp.gather(idx)
        assert np.array_equal(_np(b.frames), fr_ref[ref]), variant
        assert np.array_equal(_np(b.rewards).view(np.int64), r_ref[ref].view(np.int64)), variant
        assert np.array_equal(_np(b.terminals), d_ref[ref]) and np.array_equal(_np(b.actions), a_ref[ref]), variant
        assert np.array_equal(_np(b.boot_indices), boot_ref), variant
    # the stacks of 8 distinct frames refill K3's 4-buffer ring; repeated slots (static screens) leave U < 8
    u = [len({fr_ref[i].reshape(8, F)[j].tobytes() for j in range(8)}) for i in ref]
    assert max(u) == 8 and (min(u) < 8 or n > 4)
    x = torch.from_numpy(fr_ref[ref]).float().view((len(live), 8) + tuple(shape))
    conv = {0: x.div(255), 1: x * torch.tensor(np.float32(1.0 / 255.0)), 2: x}
    for mode, want in conv.items():
        for dt in (torch.float32, torch.bfloat16):
            b = rp.gather(idx, normalized=mode, obs_dtype=dt)
            w = want.to(dt)
            assert torch.equal(b.obs.cpu(), w[:, :4]) and torch.equal(b.next_obs.cpu(), w[:, 4:]), (mode, dt)
            assert np.array_equal(_np(b.rewards).view(np.int64), r_ref[ref].view(np.int64))
            assert np.array_equal(_np(b.boot_indices), boot_ref) and np.array_equal(_np(b.actions), a_ref[ref])


# ------------------------------------------------------------------------------------------- mailbox + waves
@pytest.mark.parametrize("Bn,k", [(32, 4), (512, 2)])
@pytest.mark.parametrize("size", ["F16", "F8192", "F25600"])
def test_mailbox_and_wave_gathers_equal_the_single_launch(size, Bn, k):
    """a0_rb_sample_gather (the gather resident under the sampler, positions through the mailbox) and the waved
    ReplayTargetLoop step (a0_rb_gather_mail per wave, ordered fetch window), eager and graph-replayed, against the
    sampler followed by one gather launch on a twin shard.  At 25 600 B the K3 ring is 100 KB, two CTAs per SM: the
    co-residence the mailbox and the fetch window rely on is at its tightest.  The fault word stays 0."""
    from agent0_b200.hotloop import ReplayTargetLoop
    shape = by_size[size]
    T = Bn * k

    def shard():
        rp = _shard(shape, 1024, 1000, n=3, algo="c51", E=8, B=Bn)
        fill_shard_synthetic(rp, 1200, 8, 3)
        ids = torch.arange(0, 1000, 7, device="cuda")
        rp.update_priority(ids, torch.rand(len(ids), device="cuda", generator=torch.Generator("cuda").manual_seed(3)) * 4)
        return rp

    o = _outputs("c51", T)
    rp_a, rp_b = shard(), shard()
    la = ReplayTargetLoop(rp_a, "c51", Bn, k, LOOP_A, o, n_step=3, rng_seed=9, gather_waves=None)
    lm = ReplayTargetLoop(rp_a, "c51", Bn, k, LOOP_A, o, n_step=3, rng_seed=9, gather_waves=None, overlap_sample_gather=True)
    lw = ReplayTargetLoop(rp_b, "c51", Bn, k, LOOP_A, o, n_step=3, rng_seed=9, gather_waves="auto", waves_when_eager=True)
    assert lw.waves is not None
    if Bn * 16 * frame_bytes(shape) >= 10_000_000:
        assert [w[1] for w in lw.waves] == [1] * k                       # one wave per batch
    draw = ("idx", "prio", "w", "frames", "act", "r64", "r32", "d8", "d32", "boot")

    def same(x, fields):
        torch.cuda.synchronize()
        for f in fields:
            assert torch.equal(getattr(la, f), getattr(x, f)), f

    rp_a.push_dynamic(); rp_b.push_dynamic()
    for call in (40, 41):                                                # the mailbox re-arms itself
        rp_a.rng_seek(call); la.sample(); la.gather()
        rp_a.rng_seek(call); lm.frames.zero_(); lm.idx.fill_(-1); lm.sample_gather()
        same(lm, draw)
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        lm.sample_gather()
    for call in (50, 51):
        rp_a.rng_seek(call); la.sample(); la.gather()
        rp_a.rng_seek(call); lm.frames.zero_(); gr.replay()
        same(lm, draw)
    full = draw + ("loss", "grad")
    rp_a.rng_seek(0); rp_b.rng_seek(0)
    for _ in range(2):
        lw.frames.zero_(); lw.idx.fill_(-1)
        la.step(); lw.step()
        same(lw, full)
        assert torch.equal(rp_a.tree, rp_b.tree)
    la.capture(warm=1); lw.capture(warm=1)
    times = []
    for _ in range(3):
        la.run()
        torch.cuda.synchronize()
        lw.frames.zero_()
        t0 = time.perf_counter()
        lw.run()
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
        same(lw, full)
        assert torch.equal(rp_a.tree, rp_b.tree)
    lib = _lib.load()
    assert lib.a0_rb_check_fault(rp_a.h) == 0 and lib.a0_rb_check_fault(rp_b.h) == 0
    print(f"\n[{size} B={Bn} k={k}] waved graph step: {min(times) * 1e6:.0f} us (best of 3, host clock around a synchronised "
          f"replay; {torch.cuda.get_device_name()})")


# ------------------------------------------------------------------------------------------------------- K6a
@pytest.mark.parametrize("shape", SHAPES, ids=IDS)
def test_decode_equals_the_oracle_at_every_frame_size(shape, k6_kernel):
    """liblz4-compressed entries (Atari-like stacks, noise, constant, a period-251 pattern), raw entries and hand-built
    blocks (overlapping matches of short periods, long runs, and far matches: offsets 65 534 / 65 535 above 64 KB,
    a match reaching back to byte 0, matches that end exactly at 8F) decode to oracle/lz4_block.py's bytes, in both
    forms of K6a.  At 16 B and 25 600 B the malformed blocks report the oracle's status."""
    F = frame_bytes(shape)
    total = 8 * F
    rp = _shard(shape, 64, 300, native=False)
    z = CP.lz4()
    rng = np.random.RandomState(F)
    s = record_stream(3, 5, seed=8, frame_hw=hw2(shape))
    fr = OR.pack_nstep(s["obs"], s["action"], s["reward"], s["done"], 3, 0.99)[0]
    plain = [fr[i].tobytes() for i in range(len(fr))]
    plain += [rng.randint(0, 256, total, dtype=np.uint8).tobytes(), bytes(total), bytes([7]) * total,
              (bytes(range(251)) * (total // 251 + 1))[:total]]
    blobs = [z.compress(p) for p in plain] + [plain[0], plain[-4]]          # raw entries, taken as they are
    for periods in ([1], [3], list(range(1, 41)), [255, 256, 257], [1, 2, 4, 7, 64, 1000, 5000]):
        blobs.append(LZ.encode_sequences(_random_sequences(rng, total, periods))[0])
    blobs += [LZ.encode_sequences(seqs)[0] for seqs, _ in far_blocks(rng, total)]
    want = [b if len(b) == total else LZ.decode(b, total) for b in blobs]
    assert want[:len(plain)] == plain
    out, status = rp.decode_entries(blobs)
    assert (status == 0).all(), status
    got = _np(out)
    for i, w in enumerate(want):
        assert got[i].tobytes() == w, f"entry {i} differs"
    if F in (16, 25600):
        check_malformed_blocks(shape)


# ------------------------------------------------------------------------------------------ K6b / K6c (extend)
@pytest.mark.parametrize("shape", SHAPES, ids=IDS)
def test_extend_labels_tell_near_identical_frames_apart(shape):
    """ReplayDataset.extend (device decode, labels, a0_ex_resolve) against the host deduper on a twin index: the same
    frame sequence numbers after every call, and every live entry gathers to its reference tuple.  The entries include
    frames that differ from an earlier frame of the same entry, or of the stream's previous entry, only in their last
    byte or only in their first byte, and frames identical to one -- the byte compare has to cover the whole frame."""
    F = frame_bytes(shape)
    E, N, NF = 4, 64, 128
    calls = (40, 7, 50, 1, 30)
    M = sum(calls)
    s = record_stream(E, M // E + 2, seed=F, frame_hw=hw2(shape), p_terminal=0.03, p_life_loss=0.04, p_truncated=0.02)
    fr, a, r, d = OR.pack_nstep(s["obs"], s["action"], s["reward"], s["done"], 1, 0.99)
    fr = fr[:M].copy()
    v = fr.reshape(M, 8, F)

    def flip(x, at):
        y = x.copy()
        y[at] ^= 0x5A
        return y

    for i in range(1 + 3 * E, M - E, 9 * E):                              # stream 1, every 9th step
        v[i, 7] = flip(v[i, 6], -1)          # last byte differs from a frame of the same entry
        v[i, 5] = flip(v[i, 6], 0)           # first byte differs
        v[i, 4] = v[i, 6]                    # identical
        v[i + E, 2] = flip(v[i, 6], -1)      # the next entry of the stream: against the previous entry's frames
        v[i + E, 1] = flip(v[i, 6], 0)
        v[i + E, 0] = v[i, 7]
    for i in range(2 + 5 * E, M, E)[:6]:
        fr[i] = np.tile(fr[2, :F], 8)                                     # static screen on stream 2
    z = CP.lz4()
    rp = _shard(shape, N, NF, native=False)
    twin = NativeRingIndex(N, rp.index.NF, 1, rp.index.age_limit)
    dd = NativeContentDeduper(twin, F)
    lo = 0
    for c in calls:
        hi = lo + c
        rp.extend([(z.compress(fr[i].tobytes()) if i % 5 else fr[i].tobytes(), a[i], r[i], d[i]) for i in range(lo, hi)],
                  streams=np.arange(lo, hi) % E)
        st = np.arange(lo, hi, dtype=np.int64) % E
        for c0 in range(0, c, twin.max_chunk):
            c1 = min(c, c0 + twin.max_chunk)
            fs8, new = dd.resolve(st[c0:c1], np.ascontiguousarray(fr[lo + c0:lo + c1].reshape(c1 - c0, 8, F)))
            twin.plan(st[c0:c1], fs8, new, a[lo + c0:lo + c1], r[lo + c0:lo + c1], d[lo + c0:lo + c1])
        assert (rp.index.head_fs, rp.index.head_q, rp.index.tail_q, rp.index.top) == (twin.head_fs, twin.head_q, twin.tail_q, twin.top)
        lo = hi
        live = np.flatnonzero(rp.index.sampleable)
        q = rp.index.head_q - 1 - ((rp.index.head_q - 1 - live) % N)
        b = rp.gather(torch.as_tensor(live, device="cuda"))
        assert np.array_equal(_np(b.frames), fr[q])
        assert np.array_equal(_np(b.actions), a[q]) and np.array_equal(_np(b.terminals), d[q])
        assert np.array_equal(_np(b.rewards).view(np.int64), r[q].view(np.int64))
    assert rp.index.head_fs > NF and rp.index.tail_q > 0                  # both rings wrapped


# ------------------------------------------------------------------------------------------------------- K7
@pytest.mark.parametrize("kind", ["noise", "constant", "synthetic", "mixed"])
@pytest.mark.parametrize("shape", SHAPES, ids=IDS)
def test_k7_equals_encode_greedy_and_the_frame_hash(shape, kind):
    """K7's blocks equal encode_greedy's, decode back through K6a, and repeat across launches; its frame hashes equal
    a0_k6_frame_hash restated in numpy (tests/frame_cases.py), partial last round of lanes included."""
    F = frame_bytes(shape)
    groups = _groups(F, kind, 3, seed=F + len(kind), hw=hw2(shape))
    blobs, hashes = encode(groups, F)
    for g, b in zip(groups, blobs):
        assert b == encode_greedy(g)
    flat = np.frombuffer(b"".join(groups), np.uint8).reshape(-1, F)
    got = [int(x) & 0xFFFFFFFFFFFFFFFF for x in hashes.tolist()]
    assert got == [frame_hash(f) for f in flat]
    dec, status = _shard(shape, 64, 300, native=False).decode_entries(blobs)
    assert (status == 0).all()
    assert dec.cpu().numpy().tobytes() == b"".join(groups)
    blobs2, hashes2 = encode(groups, F)
    assert blobs2 == blobs and torch.equal(hashes, hashes2)


# ------------------------------------------------------------------------------------------------ checkpoint
@pytest.mark.parametrize("shape", SHAPES, ids=IDS)
def test_checkpoint_round_trip(shape, tmp_path):
    """save (K7) and load (K6a, every decoded frame's hash compared with the one K7 saved) at every frame size: the
    frame ring holds Atari-like groups, a noise group (stored raw) and a last group that is not full (zero-padded);
    the loaded shard equals the saved one and stays equal under one more step of ingest, draws and updates."""
    F = frame_bytes(shape)
    E = CK_E
    src = _shard(shape, 128, 300, n=3, algo="c51", E=E, B=16)
    env = record_stream(E, 50, seed=F, frame_hw=hw2(shape))
    src.reset_streams(np.arange(E), env["obs"][0].reshape((E, 4) + tuple(shape)))
    rng = np.random.RandomState(F)
    for k in range(50):
        new = env["obs"][k + 1][:, 3].reshape((E,) + tuple(shape))
        if k == 20:
            new = rng.randint(0, 256, new.shape).astype(np.uint8)                     # with k == 21: 8 noise frames
        if k == 21:
            new = rng.randint(0, 256, new.shape).astype(np.uint8)
        src.append_steps(np.arange(E), np.ones(E, np.int64), new, env["action"][k], env["reward"][k], env["done"][k])
    extra = 3 if (src.index.head_fs + 3) % 8 else 4                                  # head_fs not a multiple of 8
    src.append_steps(np.arange(extra) % E, np.ones(extra, np.int64), rng.randint(0, 256, (extra,) + tuple(shape)).astype(np.uint8),
                     np.zeros(extra, np.int64), np.zeros(extra), np.zeros(extra, bool))
    assert src.index.head_fs % 8 != 0
    src.update_priority(torch.arange(0, 128, 3, device="cuda"), torch.linspace(0.1, 4.0, 43, device="cuda"))
    torch.cuda.synchronize()
    path = tmp_path / "shard.a0ckpt"
    src.save(path)
    dst = _shard(shape, 128, 300, n=3, algo="c51", E=E, B=16)
    dst.load(path)
    torch.cuda.synchronize()
    sa, sb = _state(src), _state(dst)
    for key in sa:
        assert (torch.equal(sa[key], sb[key]) if isinstance(sa[key], torch.Tensor) else sa[key] == sb[key]), key
    _drive([src, dst], "nstep", steps=1)


# ------------------------------------------------------------------------------ attribute caches, one process
def test_shards_of_different_frame_sizes_in_one_process():
    """The shared-memory limits of K3, the converting gather, K6a and K7 are function attributes of the process: a
    shard of 16 B frames created after one of 25 600 B must not lower the limit the first one still needs.  Order
    25 600 -> 16 (in another thread) -> 8192 -> back to the first 25 600 shard; every result against its reference."""
    def check(rp, shape, seed):
        F = frame_bytes(shape)
        rng = np.random.RandomState(seed)
        groups = [rng.randint(0, 4, 8 * F, dtype=np.uint8).tobytes(), rng.randint(0, 256, 8 * F, dtype=np.uint8).tobytes()]
        entries = np.frombuffer(b"".join(groups), np.uint8).reshape(2, 8 * F)
        rp.extend([(groups[i], i, 0.5, False) for i in range(2)], streams=np.arange(2))
        idx = torch.arange(rp.index.head_q - 2, rp.index.head_q, device="cuda") % rp.size
        for variant in (0, 2):
            rp.gather_variant = variant
            assert np.array_equal(_np(rp.gather(idx).frames), entries), variant
        b = rp.gather(idx, normalized=0)
        x = torch.from_numpy(entries.copy()).float().div(255).view((2, 8) + tuple(shape))
        assert torch.equal(b.obs.cpu(), x[:, :4]) and torch.equal(b.next_obs.cpu(), x[:, 4:])
        blobs, hashes = encode(groups, F)
        assert blobs == [encode_greedy(g) for g in groups]
        assert [int(h) & 0xFFFFFFFFFFFFFFFF for h in hashes.tolist()] == [frame_hash(f) for f in entries.reshape(16, F)]
        dec, status = rp.decode_entries(blobs)
        assert (status == 0).all() and _np(dec).tobytes() == b"".join(groups)

    big = _shard((160, 160), 64, 100, native=False)
    check(big, (160, 160), 1)
    err = []

    def small():
        try:
            check(_shard((4, 4), 64, 100, native=False), (4, 4), 2)
        except BaseException as e:          # noqa: BLE001 (re-raised in the main thread)
            err.append(e)

    t = threading.Thread(target=small)      # a record of the limits kept per thread would miss this one
    t.start(); t.join()
    if err:
        raise err[0]
    check(_shard((64, 128), 64, 100, native=False), (64, 128), 3)
    check(big, (160, 160), 4)


def test_frame_sizes_beyond_the_limit_are_refused():
    """a0_rb_create and a0_lz4_encode take F = 16 k <= 25 600: 25 616 and 7050 are refused with a message that names
    the limit, and no handle is left behind."""
    lib = _lib.load()
    for F, msg in ((25616, b"25 600"), (7050, b"multiple of 16")):
        h = C.c_void_p()
        assert lib.a0_rb_create(C.byref(h), 64, 100, F, 0) == -1 and msg in lib.a0_last_error()
        assert not h.value
        buf = torch.zeros(8 * 25616 + 64, dtype=torch.uint8, device="cuda")
        ln = torch.zeros(1, dtype=torch.int32, device="cuda")
        hs = torch.zeros(8, dtype=torch.int64, device="cuda")
        assert lib.a0_lz4_encode(buf.data_ptr(), 1, F, buf.data_ptr(), ln.data_ptr(), hs.data_ptr(), _lib.stream_ptr()) == -1
        assert msg in lib.a0_last_error()
