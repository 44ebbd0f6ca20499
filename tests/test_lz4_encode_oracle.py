"""oracle/lz4_encode.py (the specification of the device encoder K7): its blocks decode to the input under
oracle/lz4_block.py and the system liblz4, respect the block format's end rules and offset limit, and are
about as small as liblz4's own LZ4_compress_default on Atari-like frame groups.  CPU only."""
import ctypes as C

import numpy as np
import pytest

from agent0_b200.synth import SyntheticStreams
from oracle import cpu_path as CP
from oracle import lz4_block as LZ
from oracle import lz4_encode as LE
from tests.frame_cases import far_blocks, frame_bytes, hw2


def _liblz4_decode(blob, size):
    out = C.create_string_buffer(size)
    k = CP.lz4().lib.LZ4_decompress_safe(blob[4:], out, len(blob) - 4, size)
    assert k == size
    return out.raw


def _matches(blob):
    """(start, end, offset) of every match of a python-lz4 blob, and the length of the last literal run."""
    src, n = blob[4:], len(blob) - 4
    ip = op = 0
    out = []
    while True:
        tok = src[ip]; ip += 1
        ll = tok >> 4
        if ll == 15:
            while True:
                x = src[ip]; ip += 1; ll += x
                if x != 255:
                    break
        ip += ll; op += ll
        if ip >= n:
            return out, ll
        off = src[ip] | (src[ip + 1] << 8); ip += 2
        ml = tok & 15
        if ml == 15:
            while True:
                x = src[ip]; ip += 1; ml += x
                if x != 255:
                    break
        ml += 4
        out.append((op, op + ml, off))
        op += ml


def synth_groups(count, seed=0, hw=(84, 84), envs=4):
    """8-frame groups of an Atari-like frame ring: each step of ``envs`` streams appends one new frame per stream
    (four after a reset or a life loss), in ring order -- what a checkpoint of a shard encodes."""
    env = SyntheticStreams(envs, seed=seed, frame_hw=hw)
    obs, _ = env.reset()
    frames = [f for e in range(envs) for f in obs[e]]
    while len(frames) < 8 * count:
        obs, _, term, trunc, info = env.step(env.sample_actions())
        for e in range(envs):
            fresh = term[e] or trunc[e] or info["life_loss"][e]
            frames.extend(obs[e] if fresh else obs[e, 3:])
    flat = np.stack(frames[:8 * count]).reshape(count, -1)
    return [g.tobytes() for g in flat]


def _cases():
    rng = np.random.RandomState(1)
    yield "noise", rng.randint(0, 256, 56448, dtype=np.uint8).tobytes()
    yield "zeros", bytes(56448)
    yield "period3", (b"abc" * 30000)[:56448]
    yield "period84", (bytes(rng.randint(0, 256, 84, dtype=np.uint8)) * 700)[:56448]
    yield "big96", bytes(rng.randint(0, 3, 73728, dtype=np.uint8))
    for i, g in enumerate(synth_groups(3, seed=5)):
        yield f"group{i}", g
    yield "group96", synth_groups(1, seed=6, hw=(96, 96))[0]
    yield "short", b"hello world, hello world, hello world"
    yield "tiny", b"x"
    yield "f16", bytes(rng.randint(0, 2, 128, dtype=np.uint8))


@pytest.mark.parametrize("name,data", list(_cases()), ids=[c[0] for c in _cases()])
def test_encode_greedy_round_trips(name, data):
    blob = LE.encode_greedy(data)
    if len(blob) == len(data):
        assert blob == data                                   # stored raw: K6a takes it as uncompressed
        assert len(LZ.decode(len(data).to_bytes(4, "little") + LE.encode_block(data))) == len(data)
        return
    assert len(blob) < len(data)
    assert LZ.decode(blob, len(data)) == data
    assert _liblz4_decode(blob, len(data)) == data
    ms, last = _matches(blob)
    n = len(data)
    assert last >= LE.LAST_LITERALS or n < LE.MF_LIMIT
    for s, e, off in ms:
        assert s + LE.MF_LIMIT <= n and e <= n - LE.LAST_LITERALS and 1 <= off <= LE.MAX_OFFSET and e - s >= 4


def test_noise_and_zeros():
    rng = np.random.RandomState(2)
    noise = rng.randint(0, 256, 56448, dtype=np.uint8).tobytes()
    assert LE.encode_greedy(noise) == noise
    z = LE.encode_greedy(bytes(56448))
    assert len(z) < 300
    ms, last = _matches(z)
    assert ms == [(1, 56448 - 5, 1)] and last == 5                # one overlapping match up to the 5-byte limit


def test_matches_at_the_end_limits():
    rng = np.random.RandomState(3)
    for n in (40, 41, 57):
        base = bytearray(rng.randint(0, 256, n, dtype=np.uint8).tobytes())
        # a 4-byte repeat of the first word that starts exactly 12 bytes before the end is taken ...
        d = bytearray(base); d[n - 12:n - 8] = d[0:4]
        ms, _ = _matches(len(d).to_bytes(4, "little") + LE.encode_block(d))
        assert (n - 12, n - 8, n - 12) in ms
        assert LZ.decode_block(LE.encode_block(d), n) == bytes(d)
        # ... one that starts 11 bytes before the end is not
        d = bytearray(base); d[n - 11:n - 7] = d[0:4]
        ms, _ = _matches(len(d).to_bytes(4, "little") + LE.encode_block(d))
        assert all(s != n - 11 for s, _, _ in ms)
        assert LZ.decode_block(LE.encode_block(d), n) == bytes(d)
        # a repeat that runs to the end stops 5 bytes before it
        d = bytearray(base); d[n - 12:] = d[0:12]
        ms, last = _matches(len(d).to_bytes(4, "little") + LE.encode_block(d))
        assert (n - 12, n - 5, n - 12) in ms and last == 5
        assert _liblz4_decode(len(d).to_bytes(4, "little") + LE.encode_block(d), n) == bytes(d)


def test_hash_collision_keeps_the_latest_position():
    rng = np.random.RandomState(4)
    w1 = int(rng.randint(1, 2 ** 31))
    w2 = next(w for w in range(w1 + 1, w1 + 10 ** 7) if LE.hash4(w) == LE.hash4(w1))
    pad = lambda k: rng.randint(0, 256, k, dtype=np.uint8).tobytes()
    d = w1.to_bytes(4, "little") + pad(20) + w2.to_bytes(4, "little") + pad(20) + w1.to_bytes(4, "little") + pad(20)
    ms, _ = _matches(len(d).to_bytes(4, "little") + LE.encode_block(d))
    assert all(s != 48 for s, _, _ in ms)           # the table holds w2's position: w1 at 48 finds no match
    assert LZ.decode_block(LE.encode_block(d), len(d)) == d
    d2 = w1.to_bytes(4, "little") + pad(44) + w1.to_bytes(4, "little") + pad(20)
    ms, _ = _matches(len(d2).to_bytes(4, "little") + LE.encode_block(d2))
    assert ms and ms[0][0] == 48 and ms[0][2] == 48


def test_offset_limit_above_64k():
    rng = np.random.RandomState(5)
    word = rng.randint(0, 256, 16, dtype=np.uint8).tobytes()
    d = bytearray(rng.randint(0, 256, 73728, dtype=np.uint8).tobytes())
    d[0:16] = word
    d[65540:65556] = word                            # 65540 bytes back: beyond the format's offset limit
    d[70000:70016] = d[69900:69916]                  # 100 bytes back: found
    ms, _ = _matches(len(d).to_bytes(4, "little") + LE.encode_block(d))
    assert all(s != 65540 for s, _, _ in ms)
    assert any(s == 70000 and off == 100 for s, _, off in ms)
    assert _liblz4_decode(len(d).to_bytes(4, "little") + LE.encode_block(d), len(d)) == bytes(d)


@pytest.mark.parametrize("shape", [(64, 128), (16, 513), (64, 64, 3), (160, 160)], ids=["F8192", "F8208", "F12288", "F25600"])
def test_large_groups_round_trip_and_far_offsets_agree_with_liblz4(shape):
    """The references of the device LZ4 kernels in the large-group regime: 8F = 65 536 (the largest group of K7's u16
    table), 65 664, 98 304 and 204 800 bytes.  encode_greedy's blocks of Atari-like, noise and mixed groups decode to the
    input under oracle/lz4_block.py and liblz4; hand-built blocks with offsets up to 65 535 and a match that ends
    12 bytes before 8F decode identically under both; blocks whose last match ends exactly at 8F (which K6a accepts
    and liblz4 refuses) decode under the oracle."""
    F = frame_bytes(shape)
    n = 8 * F
    rng = np.random.RandomState(F)
    groups = synth_groups(2, seed=F, hw=hw2(shape))
    mixed = np.frombuffer(groups[0], np.uint8).reshape(8, F).copy()
    mixed[1::2] = rng.randint(0, 256, (4, F), dtype=np.uint8)
    groups += [mixed.tobytes(), bytes([9]) * n]
    for g in groups:
        blob = LE.encode_greedy(g)
        assert len(blob) < n
        assert LZ.decode(blob, n) == g
        assert _liblz4_decode(blob, n) == g
        assert all(1 <= off <= LE.MAX_OFFSET for _, _, off in _matches(blob)[0])
    noise = rng.randint(0, 256, n, dtype=np.uint8).tobytes()
    assert LE.encode_greedy(noise) == noise                     # stored raw
    offsets = set()
    for seqs, end_rules in far_blocks(rng, n):
        blob, want = LZ.encode_sequences(seqs)
        assert len(want) == n
        assert LZ.decode(blob, n) == want
        if end_rules:
            assert _liblz4_decode(blob, n) == want
        offsets |= {off for _, _, off in _matches(blob)[0]}
    assert max(offsets) == min(n - 4, 65535)
    if n > 65536:
        assert {65534, 65535} <= offsets


def test_size_within_ten_percent_of_liblz4_on_synthetic_groups():
    groups = synth_groups(24, seed=7)
    ours = sum(len(LE.encode_greedy(g)) for g in groups)
    ref = sum(len(CP.lz4().compress(g)) for g in groups)
    assert ours <= 1.1 * ref, (ours, ref)
