"""a0_ix_serialize / a0_ix_deserialize (the INDEX section of a shard checkpoint): an index restored into a fresh one
plans every later append exactly as its never-saved twin, through ring wrap and age-outs, for 1-step and n-step
gathering; truncated, corrupted and mismatched blobs are rejected and leave the index unchanged.  CPU only."""
import struct

import numpy as np
import pytest

from agent0_b200.ring_index import NativeRingIndex

S = 5


def _drive(indexes, rng, iters):
    """The same random multi-stream appends (uneven chunks, idle streams, 0..4 new frames) into every index."""
    for it in range(iters):
        m = int(rng.randint(1, indexes[0].max_chunk + 1))
        active = rng.choice(S, size=int(rng.randint(1, S + 1)), replace=False)
        stream = rng.choice(active, size=m).astype(np.int64)
        n_new = rng.choice([0, 1, 1, 1, 2, 4], size=m).astype(np.int64)
        action, reward, done = rng.randint(0, 18, m), rng.randn(m), rng.rand(m) < 0.1
        plans = []
        for ix in indexes:
            fs8 = ix.resolve_shift(stream, n_new)
            p = ix.plan(stream, fs8, np.arange(int(n_new.sum())), action, reward, done)
            plans.append((fs8, p.new_frame_pos, p.rec_meta, p.marks))
        for other in plans[1:]:
            for a, b in zip(plans[0], other):
                assert np.array_equal(a, b), it
        states = [(ix.head_q, ix.tail_q, ix.head_fs, ix.top) for ix in indexes]
        assert all(s == states[0] for s in states)
        assert all(np.array_equal(ix.sampleable, indexes[0].sampleable) for ix in indexes)


def _started(N, NF, n, age, seed, iters):
    ix = NativeRingIndex(N, NF, n, age)
    ix.plan(np.zeros(0, np.int64), np.zeros((0, 8), np.int64), np.arange(4 * S), [], [], [])
    for sid in range(S):
        ix.set_stack(sid, np.arange(4 * sid, 4 * sid + 4))
    _drive([ix], np.random.RandomState(seed), iters)
    return ix


@pytest.mark.parametrize("n,N,NF,age,before", [(1, 64, 300, 16, 40), (3, 48, 220, 12, 150), (4, 200, 5000, 64, 3),
                                               (2, 16, 120, 8, 200)])
def test_restored_index_plans_like_its_twin(n, N, NF, age, before):
    twin = _started(N, NF, n, age, 7 + n, before)
    blob = twin.serialize()
    loaded = NativeRingIndex(N, NF, n, age)
    loaded.deserialize(blob)
    assert loaded.serialize() == blob
    for sid in range(S):
        assert np.array_equal(loaded.get_stack(sid), twin.get_stack(sid))
    _drive([twin, loaded], np.random.RandomState(99 + n), 200)
    assert twin.tail_q > 0 and twin.serialize() == loaded.serialize()


def test_bad_blobs_are_rejected_and_leave_the_index_unchanged():
    ix = _started(64, 300, 3, 16, 11, 60)
    blob = ix.serialize()
    target = _started(64, 300, 3, 16, 12, 5)
    before = target.serialize()
    bad = [blob[:-1], blob[:100], blob + b"\0", b"XXXX" + blob[4:],
           blob[:8] + struct.pack("<q", 65) + blob[16:]]                         # another record capacity
    hq, tq, hfs, top = struct.unpack_from("<4q", blob, 40)
    bad.append(blob[:40] + struct.pack("<4q", hq, tq, hfs, top + 1) + blob[72:])    # top does not count the sampleable records
    bad.append(blob[:40] + struct.pack("<4q", tq - 1, tq, hfs, top) + blob[72:])    # head behind tail
    samp_at = 72 + 64 * 8
    flip = bytearray(blob)
    q = next(i for i in range(64) if flip[samp_at + i] == 0 and not (tq % 64 <= i < tq % 64 + (hq - tq)))
    flip[samp_at + q] = 1                                                        # a dead record marked sampleable
    bad.append(bytes(flip))
    flip = bytearray(blob)
    flip[samp_at + 64 + 8 + 16] ^= 0x01                                          # stream 0's last_seq
    bad.append(bytes(flip))
    for b in bad:
        with pytest.raises(RuntimeError):
            target.deserialize(b)
        assert target.serialize() == before
    with pytest.raises(RuntimeError, match="N=64"):
        NativeRingIndex(64, 300, 1, 16).deserialize(blob)
    with pytest.raises(RuntimeError, match="NF=300"):
        NativeRingIndex(64, 400, 3, 16).deserialize(blob)
