"""K6 on the GPU through the C ABI: the LZ4 block decoder (a0_ex_decode) bit-exact against
oracle/lz4_block.py (itself pinned to liblz4 in tests/test_lz4_oracle.py), its status codes on malformed
blocks, and ReplayDataset.extend end to end -- the device de-duplication must take the decisions of the
host specification (a0_dd_resolve) and every gathered entry must equal the reference entry, bit for bit."""
import numpy as np
import pytest
import torch

from agent0_b200.config import make_config
from agent0_b200.ring_index import NativeContentDeduper, NativeRingIndex
from agent0_b200.synth import record_stream
from oracle import cpu_path as CP
from oracle import lz4_block as LZ
from oracle import reference_replay as OR

pytestmark = pytest.mark.gpu


def _np(t):
    return t.detach().cpu().numpy()


def _replay(size, hw=(84, 84), E=4, per=True, **kw):
    from agent0_b200.replay import ReplayDataset
    cfg = make_config("c51", per=per, n_step=3, batch_size=8, replay_size=size, num_envs=E)
    cfg.obs_shape = (4,) + tuple(hw)
    cfg.trainer.total_steps = 100000
    return ReplayDataset(cfg, **kw)


def _random_sequences(rng, total, periods):
    """Sequences whose decoded length is exactly ``total``: random literal runs and matches with the
    given offsets (periods), lengths around the 15 / 19 / 255-chain boundaries."""
    seqs, n = [], 0
    lens = [4, 5, 18, 19, 20, 60, 127, 128, 129, 273, 274, 275, 529, 1000]
    while True:
        ll = int(rng.choice([0, 1, 3, 14, 15, 16, 40, 127, 128, 129, 269, 270, 271, 600]))
        if n == 0:
            ll = max(ll, 1)
        off = int(rng.choice(periods))
        ml = int(rng.choice(lens))
        if n + ll + ml + 16 > total:
            break
        lit = rng.randint(0, 256, ll, dtype=np.uint8).tobytes()
        if off > n + ll:
            off = max(1, n + ll)
        seqs.append((lit, off, ml))
        n += ll + ml
    seqs.append((rng.randint(0, 256, total - n, dtype=np.uint8).tobytes(), None, None))
    return seqs


A0_OPT_K6_GLOBAL = 11


@pytest.fixture(params=[0, 1], ids=["shared_memory", "in_place"])
def k6_kernel(request):
    """Both forms of the decode kernel: output staged in shared memory (default) and decoded in place in the scratch."""
    from agent0_b200 import _lib
    _lib.check(_lib.load().a0_set_option(A0_OPT_K6_GLOBAL, request.param), "a0_set_option")
    yield request.param
    _lib.check(_lib.load().a0_set_option(A0_OPT_K6_GLOBAL, 0), "a0_set_option")


@pytest.mark.parametrize("hw", [(84, 84), (16, 16), (8, 8)])
def test_decode_equals_the_oracle(hw, k6_kernel):
    """liblz4-compressed entries (synthetic Atari-like stacks, noise, constant screens) and hand-built
    blocks -- overlapping matches of every period 1..40 and beyond, long literal and match runs, length
    fields on every extension boundary, raw (uncompressed) entries -- decode to the oracle's bytes."""
    F = hw[0] * hw[1]
    total = 8 * F
    rp = _replay(64, hw=hw)
    z = CP.lz4()
    rng = np.random.RandomState(5)
    s = record_stream(3, 12, seed=8, frame_hw=hw)
    fr, _, _, _ = OR.pack_nstep(s["obs"], s["action"], s["reward"], s["done"], 3, 0.99)
    plain = [fr[i].tobytes() for i in range(len(fr))]
    plain += [rng.randint(0, 256, total, dtype=np.uint8).tobytes(), bytes(total), bytes([7]) * total,
              (bytes(range(251)) * (total // 251 + 1))[:total]]
    blobs, want = [], []
    for p in plain:
        blobs.append(z.compress(p)); want.append(p)
    blobs.append(plain[0]); want.append(plain[0])                       # raw entry, taken as it is
    for periods in ([1], [2], [3], [4], list(range(1, 41)), [31, 32, 33], [255, 256, 257, 300], [1, 2, 4, 7, 64, 1000, 5000]):
        for _ in range(3):
            blob, w = LZ.encode_sequences(_random_sequences(rng, total, periods))
            assert LZ.decode(blob, total) == w
            blobs.append(blob); want.append(w)
    out, status = rp.decode_entries(blobs)
    assert (status == 0).all(), status
    got = _np(out)
    for i, w in enumerate(want):
        assert got[i].tobytes() == w, f"entry {i} differs"


def test_decode_keeps_working_after_a_shard_of_smaller_frames():
    """K6a's shared-memory limit is an attribute of the kernel for the whole process: a shard of 16-byte frames must not
    lower it under a shard of 84x84 frames created earlier (a per-shard 'already set' flag did, and the earlier
    shard's next decode failed to launch)."""
    z = CP.lz4()
    rng = np.random.RandomState(3)
    blobs = {}
    for hw in ((84, 84), (4, 4)):
        p = rng.randint(0, 4, 8 * hw[0] * hw[1], dtype=np.uint8).tobytes()
        blobs[hw] = (z.compress(p), p)
    big = _replay(64, hw=(84, 84))
    for rp, hw in ((big, (84, 84)), (_replay(64, hw=(4, 4)), (4, 4)), (big, (84, 84))):
        out, status = rp.decode_entries([blobs[hw][0]])
        assert (status == 0).all() and _np(out)[0].tobytes() == blobs[hw][1]


def test_decode_reports_malformed_blocks(k6_kernel):
    check_malformed_blocks((8, 8))


def check_malformed_blocks(hw):
    """Truncated blocks, a wrong size prefix, offsets past what has been produced or 0, blocks that decode to more or
    fewer than 8 frames: K6a reports the oracle's status, and extend() refuses the call and commits nothing."""
    total = 8 * int(np.prod(hw))
    rp = _replay(64, hw=hw)
    rng = np.random.RandomState(2)
    seqs = _random_sequences(rng, total - 12, [1, 5, 40])
    good, want = LZ.encode_sequences([(b"abcdefgh", 3, 4)] + seqs)      # a first sequence with a short literal run
    bad = [good, good[:len(good) // 2], (total + 16).to_bytes(4, "little") + good[4:], b"\x00\x02\x00", good[:4]]
    b2 = bytearray(good)
    # first sequence: token, literals, offset -> an offset larger than what has been produced
    ll = b2[4] >> 4
    assert ll < 15
    b2[4 + 1 + ll] = 0xff; b2[4 + 2 + ll] = 0xff
    bad.append(bytes(b2))
    b3 = bytearray(good); b3[4 + 1 + ll] = 0; b3[4 + 2 + ll] = 0
    bad.append(bytes(b3))
    long_, _ = LZ.encode_sequences([(b"abcdefgh", 8, total), (b"", None, None)], size=total)
    short, _ = LZ.encode_sequences([(b"abcdefgh", 8, 4), (b"", None, None)], size=total)
    bad += [long_, short]
    out, status = rp.decode_entries(bad)
    expect = [LZ.status(b, total) for b in bad]
    assert expect[0] == 0 and all(e != 0 for e in expect[1:])
    assert status.tolist() == expect
    assert _np(out)[0].tobytes() == want
    # extend() refuses the call and commits nothing
    with pytest.raises(RuntimeError, match="not a valid lz4 block"):
        rp.extend([(good, 0, 0.0, False), (short, 0, 0.0, False)])
    assert rp.top == 0 and rp.index.head_fs == 0
    rp.extend([(good, 1, 0.5, False)])
    assert rp.top == 1


@pytest.mark.parametrize("n,N,age,calls", [(3, 4096, None, (1280, 640, 37, 1, 300)), (1, 96, 12, (50, 7, 120, 33, 200, 64)),
                                          (3, 8192, None, (2500, 100))])      # 2500 > 2048: two decode batches inside one call
def test_extend_takes_the_decisions_of_the_host_deduper(n, N, age, calls):
    """The same lz4 entries through ReplayDataset.extend (device decode + labels + a0_ex_resolve) and
    through the host specification (liblz4 decode + a0_dd_resolve + a0_ix_plan on a twin index): the same
    frame sequence numbers, so the same ring contents; every live entry gathers to the reference entry.
    Includes static screens, repeats inside an entry, ring wrap and frames that age out."""
    E = 4
    hw = (84, 84) if N > 1000 else (16, 16)
    F = hw[0] * hw[1]
    M = sum(calls)
    s = record_stream(E, M // E + n + 2, seed=21 + n, frame_hw=hw, p_terminal=0.03, p_life_loss=0.04, p_truncated=0.02)
    fr, a, r, d = OR.pack_nstep(s["obs"], s["action"], s["reward"], s["done"], n, 0.99)
    fr = fr[:M].copy()
    for i in range(1 + 5 * E, M, E)[:9]:
        fr[i] = np.tile(fr[1, :F], 8)                                     # static screen on stream 1
    fr[2 + 9 * E].reshape(8, F)[5] = fr[2 + 9 * E].reshape(8, F)[0]         # a frame repeated inside one entry
    z = CP.lz4()
    NF = 4 * N + 64 if N < 65536 else None
    rp = _replay(N, hw=hw, E=E, frame_capacity=NF, age_limit=age)
    twin = NativeRingIndex(N, rp.index.NF, 1, age)
    dd = NativeContentDeduper(twin, F)
    lo = 0
    for c in calls:
        hi = lo + c
        tup = [(z.compress(fr[i].tobytes()) if i % 5 else fr[i].tobytes(), a[i], r[i], d[i]) for i in range(lo, hi)]
        rp.extend(tup, streams=np.arange(lo, hi) % E)
        st = np.arange(lo, hi, dtype=np.int64) % E
        for c0 in range(0, c, twin.max_chunk):
            c1 = min(c, c0 + twin.max_chunk)
            fs8, new = dd.resolve(st[c0:c1], np.ascontiguousarray(fr[lo + c0:lo + c1].reshape(c1 - c0, 8, F)))
            twin.plan(st[c0:c1], fs8, new, a[lo + c0:lo + c1], r[lo + c0:lo + c1], d[lo + c0:lo + c1])
        assert (rp.index.head_fs, rp.index.head_q, rp.index.tail_q, rp.index.top) == (twin.head_fs, twin.head_q, twin.tail_q, twin.top)
        lo = hi
        live = np.flatnonzero(rp.index.sampleable)
        q = rp.index.head_q - 1 - ((rp.index.head_q - 1 - live) % N)        # entry held by each live ring position
        b = rp.gather(torch.as_tensor(live, device="cuda"))
        assert np.array_equal(_np(b.frames), fr[q])
        assert np.array_equal(_np(b.actions), a[q]) and np.array_equal(_np(b.terminals), d[q])
        assert np.array_equal(_np(b.rewards).view(np.int64), r[q].view(np.int64))
    if age is None:
        assert rp.index.head_fs < 3 * M                                    # ~1-2 stored frames per entry, not 8
    t = rp.extend_timing()
    assert t["entries"] == calls[-1] and t["device_decode_label_us"] > 0


def test_extend_rejects_native_nstep_shards():
    """Reference entries are already n-step folded: a shard that folds again at gather time must refuse them."""
    from agent0_b200.replay import ReplayDataset
    cfg = make_config("c51", per=True, n_step=3, batch_size=8, replay_size=64, num_envs=2)
    rp = ReplayDataset(cfg, native_nstep=True)
    with pytest.raises(RuntimeError, match="n-step"):
        rp.extend([(bytes(8 * 7056), 0, 0.0, False)])
