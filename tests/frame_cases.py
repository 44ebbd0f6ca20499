"""Frame sizes the C ABI accepts (F a positive multiple of 16 with 8F <= 200 KB) and the pieces the frame-size tests
share: hand-built LZ4 blocks whose matches reach the format's offset limit, and the frame hash of K6a / K7 restated
in numpy.  Test infrastructure only."""
import numpy as np

# (frame shape, why).  F = prod(shape).
SIZES = [
    ((4, 4), "one 16-byte vector: a single hash lane, 4 f32 groups, 2 bf16 groups"),
    ((4, 12), "not a multiple of 32 or 64"),
    ((16, 31), "31 vectors: one hash lane idle"),
    ((16, 32), "exactly 32 vectors"),
    ((84, 84), "the Atari frame"),
    ((64, 128), "8F = 65 536: the largest group of K7's u16 table; offsets reach every byte"),
    ((16, 513), "8F = 65 664: the first group of K7's u32 table"),
    ((64, 64, 3), "64x64 RGB"),
    ((128, 128), "16 384"),
    ((16, 1599), "25 584: the largest size below the limit that is not a round number"),
    ((160, 160), "25 600: the limit, 200 KB groups"),
]
SHAPES = [s for s, _ in SIZES]
IDS = ["F%d" % int(np.prod(s)) for s in SHAPES]


def frame_bytes(shape):
    return int(np.prod(shape))


def hw2(shape):
    """A 2-D (h, w) with the same byte count, for the synthetic Atari-like stream generators."""
    return (int(shape[0]), frame_bytes(shape) // int(shape[0]))


def far_blocks(rng, total):
    """[(sequences, end_rules)]: sequences [(literals, offset, match length) ..., (literals, None, None)] for
    oracle.lz4_block.encode_sequences that decode to exactly ``total`` bytes.  A match that ends exactly at ``total``
    with the longest offset the block allows (back to byte 0 when total <= 65 539): K6a and the oracle take it, but it
    breaks the block format's end rules (the last 5 bytes are literals), which liblz4 enforces (end_rules False).  The
    same far match ending 12 bytes early, and, from 8F = 65 664 up, matches at offsets 65 535 and 65 534 (end_rules
    True: liblz4 decodes them too)."""
    lit = lambda k: rng.randint(0, 256, k, dtype=np.uint8).tobytes()
    a = min(total - 4, 65535)
    out = [([(lit(a), a, total - a), (b"", None, None)], False)]
    a = min(total - 16, 65535)
    out.append(([(lit(a), a, total - a - 12), (lit(12), None, None)], True))
    if total >= 65664:
        seqs = [(lit(65535), 65535, 16), (lit(1), 65534, 20), (lit(5), 65535, 4)]
        rest = total - sum(len(s[0]) + s[2] for s in seqs)
        out.append((seqs + [(lit(rest - 60), 65535, 40), (lit(20), None, None)], True))
        out.append((seqs + [(lit(rest - 40), 65534, 40), (b"", None, None)], False))
    return out


_M32 = 0xFFFFFFFF


def _rotl(x, r):
    return ((x << np.uint64(r)) | (x >> np.uint64(32 - r))) & np.uint64(_M32)


def _mix32(h):
    h = h ^ (h >> np.uint64(16)); h = (h * np.uint64(0x85EBCA6B)) & np.uint64(_M32)
    h = h ^ (h >> np.uint64(13)); h = (h * np.uint64(0xC2B2AE35)) & np.uint64(_M32)
    return h ^ (h >> np.uint64(16))


def frame_hash(frame):
    """a0_k6_frame_hash (a0_common.cuh) of one frame: lane i of a warp folds 16-byte vectors i, i + 32, ... into four
    32-bit multiply-rotate streams; the lanes' mixed results are xor-reduced.  Returns an unsigned 64-bit int."""
    v = np.frombuffer(bytes(frame), dtype="<u4").reshape(-1, 4).astype(np.uint64)
    lane = np.arange(32, dtype=np.uint64)
    K = [0x9E3779B1, 0x85EBCA77, 0xC2B2AE3D, 0x27D4EB2F]
    R = [13, 15, 17, 11]
    h = [(np.uint64(K[c]) * (lane + np.uint64(1 + 32 * c))) & np.uint64(_M32) for c in range(4)]
    for r0 in range(0, len(v), 32):
        blk = v[r0:r0 + 32]
        k = len(blk)                                   # the last round may leave lanes idle
        for c in range(4):
            h[c][:k] = _rotl(((h[c][:k] ^ blk[:, c]) * np.uint64(K[c])) & np.uint64(_M32), R[c])
    lo = _mix32((h[0] + np.uint64(0x165667B1) * h[2]) & np.uint64(_M32))
    hi = _mix32((h[1] + np.uint64(0x9E3779B1) * h[3]) & np.uint64(_M32))
    lo = np.bitwise_xor.reduce(lo)
    hi = np.bitwise_xor.reduce(hi)
    return (int(_mix32(hi ^ np.uint64(0x5BD1E995))) << 32) | int(_mix32(lo))
