"""K9 (csrc/a0_inbox.cu, agent0_b200/inbox.py) at the shapes where its code has branches and boundaries.

1. Every frame size of tests/frame_cases.py (n = 3; n = 1 and n = A0_MAX_NSTEP at 16 B and 25 600 B): writers on
   2-3 lanes append ragged streams (static screens, whole new stacks, dones; rewards of -0.0, subnormals and +-1e300)
   and the inbox is drained at irregular points until the record ring and the frame ring have wrapped, with an age
   limit that evicts.  The shard equals (a) a twin fed the same steps in drain order with append_vector_step, and (b)
   the oracle's actor packer (oracle.reference_replay.pack_nstep) record by record through an owner map.
2. K9a and K9b against host bytes: commits of exactly 64 KB, 64 KB +- 16 B, 9 chunks + 16 B, metadata only and
   T = 1.  A commit writes the header from its arguments and the staging bytes it owns, nothing else; a scan copies
   the header and the 16-byte-rounded used prefix of every array, nothing else; bytes of a slot beyond its used
   prefixes (a smaller commit into a reused slot included) do not change what a drain ingests.
3. Slot and lane geometry: 1, 3, 5 and 64 slots with more than ten laps of the lane counters, 1024 lanes of one
   stream, a new writer of a lane resetting its streams, and a0_tx_scan / a0_tx_release called directly.
4. A slot of one vector step takes a writer's first step of whole new stacks on every stream, and a slot that
   cannot take every vector step is refused when the inbox is made.
Every comparison is bit for bit."""
import numpy as np
import pytest
import torch

from agent0_b200 import _lib
from agent0_b200.inbox import TransitionInbox, TransitionWriter
from agent0_b200.ring_index import stack_delta
from oracle import reference_replay as OR
from tests.frame_cases import IDS, SHAPES, frame_bytes
from tests.test_gpu_edges import _stream
from tests.test_gpu_frame_sizes import _shard
from tests.test_gpu_inbox import _assert_same, _state

pytestmark = pytest.mark.gpu

CHUNK = 64 * 1024                     # bytes one K9a CTA copies
SPECIAL = np.array([-0.0, 5e-324, -5e-324, 2.5e-310, 1e300, -1e300])
_ESZ = dict(step_count=8, step_reset=1, stream=8, n_new=8, action=8, reward=8, done=1)
_BY_STEPS = ("step_count", "step_reset")        # sized by vector steps; the other arrays by transitions


def _rewards(rng, shape):
    r = rng.randn(*shape)
    pick = rng.rand(*shape) < 0.3
    r[pick] = SPECIAL[rng.randint(0, len(SPECIAL), int(pick.sum()))]
    return r


def _lane_data(E, T, shape, seed):
    """T vector steps of E ragged streams (tests/test_gpu_edges._stream) with special rewards mixed in."""
    obs, n_new, act, _, done = _stream(E, T, shape, seed, p_new4=0.15, p_static=0.2)
    return obs, n_new, act, _rewards(np.random.RandomState(seed + 1), (T, E)), done


class _Lanes:
    """In-process writers on the lanes of an inbox, and what each drain must ingest: ``order`` lists (lane, data,
    step) in drain order (lane by lane, each lane's committed steps in order)."""

    def __init__(self, inbox):
        self.inbox, self.E = inbox, inbox.E
        self.writers, self.packed = {}, {}
        self.committed = {l: [] for l in range(inbox.lanes)}
        self.order = []

    def open(self, lane):
        self.writers[lane] = TransitionWriter(self.inbox, lane=lane, timeout=5.0)
        self.packed[lane] = []

    def append(self, lane, data, k):
        w, p = self.writers[lane], self.packed[lane]
        obs, _, act, rew, done = data
        w.append_vector_step(obs[k], act[k], rew[k], done[k], obs[k + 1])
        p.append((data, k))
        cut = len(p) - w.packer.n_steps                  # the steps before the packed ones are committed
        self.committed[lane] += p[:cut]
        del p[:cut]

    def flush(self, lane):
        self.writers[lane].flush()
        self.committed[lane] += self.packed[lane]
        self.packed[lane] = []

    def abandon(self, lane):
        """The lane's writer stops as if its process died: the steps it packed are lost, its slots stay committed."""
        self.packed[lane] = []
        return self.writers.pop(lane)

    def close(self, lane):
        self.writers.pop(lane).close()

    def drain(self):
        got, want = self.inbox.drain(), 0
        for l, steps in self.committed.items():
            self.order += [(l, d, k) for d, k in steps]
            want += self.E * len(steps)
            self.committed[l] = []
        assert got == want
        return got


def _drive(inbox, data, rng, max_gap):
    """Writers on every lane append the lanes' steps (data[l]), interleaved step by step; the inbox is drained after
    every 1..max_gap steps (max_gap <= slots * steps per slot: a writer never waits).  Returns the drain order."""
    lanes = _Lanes(inbox)
    for l in range(inbox.lanes):
        lanes.open(l)
    T = len(data[0][1])
    at = rng.randint(1, max_gap + 1)
    for k in range(T):
        for l in range(inbox.lanes):
            lanes.append(l, data[l], k)
        if k + 1 == at:
            lanes.drain()
            at += rng.randint(1, max_gap + 1)
    lanes.drain()                                        # the flushes below may each need a slot
    for l in range(inbox.lanes):
        lanes.flush(l)
    lanes.drain()
    assert inbox.drain() == 0
    for l in range(inbox.lanes):
        lanes.close(l)
    return lanes.order


def _feed_twin(twin, E, order):
    """Reference (a): the steps in drain order through append_vector_step, stream ids offset by lane * E; a
    writer's first step resets its streams."""
    started = set()
    for l, data, k in order:
        obs, _, act, rew, done = data
        streams = np.arange(E) + l * E
        if id(data) not in started:
            started.add(id(data))
            assert k == 0
            twin.reset_streams(streams, obs[0])
        twin.append_vector_step(obs[k], act[k], rew[k], done[k], obs[k + 1], streams=streams)


def _same_as_twin(rp, twin, what):
    """_assert_same once the frame ring has wrapped: a0_rb_create does not clear the ring, so a row neither shard has
    written yet holds whatever its allocation held."""
    assert rp.index.head_fs > rp.index.NF, f"{what}: the frame ring has not wrapped"
    _assert_same(_state(rp), _state(twin), what)


def _check_against_packer(rp, E, n, order):
    """Reference (b): every sampleable record gathers to its entry of pack_nstep over its lane's steps (frames, float64
    return bits, action, done) and to the boot index of its stream's n-th successor.  One data sequence per lane."""
    N, hist, owner, data, q = rp.size, {}, {}, {}, 0
    for l, d, k in order:
        assert data.setdefault(l, d) is d
        for e in range(E):
            owner[q % N] = (l, e, k)
            hist.setdefault((l, e), []).append(q % N)
            q += 1
    assert rp.index.head_q == q
    live = np.flatnonzero(rp.index.sampleable)
    assert len(live) == rp.top > 10
    packs = {l: OR.pack_nstep(d[0], d[2], d[3], d[4], n, rp.gamma) for l, d in data.items()}
    fr, act, rew, done, boot = [], [], [], [], []
    for p in live:
        l, e, k = owner[p]
        i = (k + n - 1) * E + e
        fr.append(packs[l][0][i]); act.append(packs[l][1][i]); rew.append(packs[l][2][i]); done.append(packs[l][3][i])
        h = hist[(l, e)]
        boot.append(h[k + n] if k + n < len(h) else -1)
    b = rp.gather(torch.as_tensor(live, device=rp.device))
    assert np.array_equal(b.frames.cpu().numpy(), np.stack(fr))
    assert np.array_equal(b.rewards.cpu().numpy().view(np.int64), np.array(rew, dtype=np.float64).view(np.int64))
    assert np.array_equal(b.actions.cpu().numpy(), np.array(act))
    assert np.array_equal(b.terminals.cpu().numpy(), np.array(done))
    assert np.array_equal(b.boot_indices.cpu().numpy(), np.array(boot))


# ------------------------------------------------------------------------------------- 1. every frame size
NMAX = _lib.A0_MAX_NSTEP
GEOMETRY = {1: (3, 3, 40, 96), 3: (3, 3, 40, 96), NMAX: (2, 2, 90, 128)}    # n -> lanes, streams per lane, steps, N
CROSSINGS = [(s, 3) for s in SHAPES] + [(s, n) for s in (SHAPES[0], SHAPES[-1]) for n in (1, NMAX)]
CROSSING_IDS = [f"{IDS[SHAPES.index(s)]}-n{n}" for s, n in CROSSINGS]


@pytest.mark.parametrize("shape,n", CROSSINGS, ids=CROSSING_IDS)
def test_every_frame_size_drains_to_the_twin_and_the_packer(shape, n):
    """K1 reads each step's frames in place at slot_frames + frame_off * F (every 16-byte residue mod 256 at small F,
    only some at 7056), reset stacks first; three vector steps per slot, three slots per lane."""
    F = frame_bytes(shape)
    lanes, E, T, N = GEOMETRY[n]
    NF, age, S, per_slot = 200, 25, 3, 3
    rp, twin = (_shard(shape, N, NF, n=n, E=E, age_limit=age) for _ in range(2))
    inbox = TransitionInbox(rp, lanes, slots=S, slot_transitions=per_slot * E)
    data = [_lane_data(E, T, shape, seed=F + 7 * n + l) for l in range(lanes)]
    order = _drive(inbox, data, np.random.RandomState(F + n), max_gap=S * per_slot)
    assert rp.index.head_q > N and rp.index.tail_q > 0                    # the record ring wrapped
    _feed_twin(twin, E, order)
    _same_as_twin(rp, twin, f"F={F} n={n}")
    _check_against_packer(rp, E, n, order)


# ----------------------------------------------------------------------------- 2. K9a and K9b against host bytes
def _used(L, n_t, n_s):
    """(offset, bytes) of the header's counts and of the used prefix of every metadata array of a slot."""
    return [(0, 24)] + [(L[k], esz * (n_s if k in _BY_STEPS else n_t)) for k, esz in _ESZ.items()]


def _scan(inbox, max_slots, heads):
    """a0_tx_scan(max_slots_per_lane=max_slots) into poisoned host memory.  Lane l's head must read heads[l] =
    (consumed, committed, taken); its entry j the 256-byte header and the 16-byte-rounded used prefix of every array of
    slot (consumed + j) % S, and nothing else of the lane's entries may be written."""
    L, S, scan = inbox.layout, inbox.slots, inbox._scan
    scan[:] = 0xA5
    with torch.cuda.device(inbox.device):
        _lib.check(inbox.lib.a0_tx_scan(inbox._h, max_slots, _lib.stream_ptr(inbox.device)), "a0_tx_scan")
        torch.cuda.current_stream(inbox.device).synchronize()
    head = scan[:32 * inbox.lanes].view(np.int64).reshape(inbox.lanes, 4)
    for l, (consumed, committed, taken) in enumerate(heads):
        assert [int(x) for x in head[l]] == [consumed, committed, taken, 0], l
        for j in range(S):
            at = L["scan_meta"] + (l * S + j) * L["frames"]
            want = np.full(L["frames"], 0xA5, dtype=np.uint8)
            if j < taken:
                sb = inbox.slot_bytes(l, (consumed + j) % S)[:L["frames"]].cpu().numpy()
                n_t, n_s = (int(x) for x in sb[:16].view(np.int64))
                want[:256] = sb[:256]
                for off, nb in _used(L, n_t, n_s)[1:]:
                    nb = -(-nb // 16) * 16
                    want[off:off + nb] = sb[off:off + nb]
            assert np.array_equal(scan[at:at + L["frames"]], want), (l, j)


def _poison_unused(inbox, lane, slot, rng):
    """Random bytes everywhere in the slot but its header's counts, the used prefixes of its arrays and its frames."""
    L = inbox.layout
    sb = inbox.slot_bytes(lane, slot)
    host = sb.cpu().numpy().copy()
    n_t, n_s, n_f = (int(x) for x in host[:24].view(np.int64))
    keep = np.zeros(len(host), dtype=bool)
    for off, nb in _used(L, n_t, n_s):
        keep[off:off + nb] = True
    keep[L["frames"]:L["frames"] + n_f * inbox.F] = True
    host[~keep] = rng.randint(0, 256, int((~keep).sum()), dtype=np.uint8)
    sb.copy_(torch.from_numpy(host))


def _split(rng, m, total):
    """m values in [0, 4] (zeros and fours included) that sum to total."""
    assert 0 <= total <= 4 * m
    v = rng.randint(0, 5, m)
    while v.sum() != total:
        d = int(total - v.sum())
        can = np.flatnonzero(v < 4) if d > 0 else np.flatnonzero(v > 0)
        v[rng.choice(can, min(abs(d), len(can)), replace=False)] += 1 if d > 0 else -1
    return v


def _pack(packer, rng, E, n_frames, reset):
    """Packs vector steps of E streams holding n_frames frames into the writer's staging (the first step resets the
    streams when ``reset``).  Returns them as (reset, n_new, action, reward, done, frames)."""
    new = n_frames - (4 * E if reset else 0)
    k = rng.randint(max(1, -(-new // (4 * E))), packer.T // E + 1)
    m = k * E
    n_new, act = _split(rng, m, new), rng.randint(0, 18, m)
    rew, done = _rewards(rng, (m,)), rng.rand(m) < 0.15
    frames = rng.randint(0, 256, (n_frames, packer.F), dtype=np.uint8)
    steps, f = [], 0
    for s in range(k):
        sl = slice(s * E, (s + 1) * E)
        r = reset and s == 0
        c = 4 * E * r + int(n_new[sl].sum())
        packer.add(r, np.arange(E), n_new[sl], act[sl], rew[sl], done[sl], frames[f:f + c])
        steps.append((r, n_new[sl], act[sl], rew[sl], done[sl], frames[f:f + c]))
        f += c
    assert f == n_frames
    return steps


# case -> streams per lane E, slot_transitions T, slots, the bytes each commit copies after the slot header (a
# function of the metadata bytes `m`, which every commit copies whole)
COMMITS = {
    "64KB": (64, 1024, 2, lambda m: [CHUNK, CHUNK + 16, CHUNK - 16, m, CHUNK, m, CHUNK + 16]),
    "9x64KB+16": (1024, 8192, 1, lambda m: [9 * CHUNK + 16, m, 8 * CHUNK]),
    "T1": (1, 1, 3, lambda m: [m + 16 * k for k in (8, 0, 1, 4, 0, 4, 1, 0, 4, 4, 1)]),
}


@pytest.mark.parametrize("case", list(COMMITS))
def test_commit_and_scan_copy_exactly_their_bytes(case):
    E, T, S, sizes = COMMITS[case]
    N, NF, age = {"64KB": (2048, 4096, None), "9x64KB+16": (16384, 20000, None), "T1": (8, 24, 4)}[case]
    shape = (4, 4)                                                           # F = 16: one frame, one vector
    rp, twin = (_shard(shape, N, NF, n=3, E=E, age_limit=age) for _ in range(2))
    inbox = TransitionInbox(rp, 1, slots=S, slot_transitions=T)
    L = inbox.layout
    meta = L["frames"] - 256
    w = TransitionWriter(inbox, lane=0, timeout=5.0)
    words = inbox.lane_words(0)
    rng = np.random.RandomState(len(case))
    gen = torch.Generator().manual_seed(len(case))
    pending = []

    def drain():
        consumed, committed = int(words[2]), int(words[1])
        for slot, _ in pending:
            _poison_unused(inbox, 0, slot, rng)
        _scan(inbox, S, [(consumed, committed, committed - consumed)])        # poison is not copied
        want = 0
        for _, steps in pending:
            for r, n_new, a, rw, d, fr in steps:
                if r:
                    twin.reset_streams(np.arange(E), fr[:4 * E])
                    fr = fr[4 * E:]
                twin.append_steps(np.arange(E), n_new, fr, a, rw, d)
                want += E
        assert inbox.drain() == want
        pending.clear()

    for i, nbytes in enumerate(sizes(meta)):
        assert (nbytes - meta) % 16 == 0
        nf = (nbytes - meta) // 16
        committed, consumed = int(words[1]), int(words[2])
        if committed - consumed == S:
            drain()
            consumed = committed
        slot = committed % S
        sb = inbox.slot_bytes(0, slot)
        sb.copy_(torch.randint(0, 256, sb.shape, dtype=torch.uint8, generator=gen))
        before = sb.cpu()
        steps = _pack(w.packer, rng, E, nf, reset=i == 0 or (nf >= 8 * E and rng.rand() < 0.5))
        n_t, n_s = w.packer.n_transitions, w.packer.n_steps
        assert w.packer.nbytes() == 256 + nbytes
        staging = w._host[:256 + nbytes].clone()
        w.flush()
        after = sb.cpu()
        assert after[:24].view(torch.int64).tolist() == [n_t, n_s, nf], "header"
        assert torch.equal(after[24:256], before[24:256]), "the header's other bytes are not the commit's"
        assert torch.equal(after[256:256 + nbytes], staging[256:]), "the committed bytes differ from the staging"
        assert torch.equal(after[256 + nbytes:], before[256 + nbytes:]), "bytes past the commit were written"
        pending.append((slot, steps))
        _scan(inbox, S, [(consumed, committed + 1, committed + 1 - consumed)])
    drain()
    assert inbox.drain() == 0
    w.close()
    _same_as_twin(rp, twin, case)


# ------------------------------------------------------------------------------------ 3. slot and lane geometry
@pytest.mark.parametrize("S,steps", [(1, 24), (3, 40), (5, 60), (64, 150)])
def test_slot_counts_and_laps_of_the_lane_counters(S, steps):
    """One vector step per slot: slot q lives at q % S for S = 1, 3, 5 (more than ten laps) and 64 (a drain takes up
    to every slot of a lane)."""
    shape, E, lanes = (4, 4), 2, 2
    rp, twin = (_shard(shape, 64, 100, n=3, E=E, age_limit=20) for _ in range(2))
    inbox = TransitionInbox(rp, lanes, slots=S, slot_transitions=E)
    data = [_lane_data(E, steps, shape, seed=10 * S + l) for l in range(lanes)]
    order = _drive(inbox, data, np.random.RandomState(S), max_gap=S)
    for l in range(lanes):
        assert [int(x) for x in inbox.lane_words(l)[1:]] == [steps, steps]
    assert S not in (3, 5) or steps > 10 * S
    _feed_twin(twin, E, order)
    _same_as_twin(rp, twin, f"{S} slots")
    _check_against_packer(rp, E, 3, order)


def test_1024_lanes_of_one_stream():
    shape, E, lanes, steps = (4, 4), 1, 1024, 5
    rp, twin = (_shard(shape, 4096, 8192, n=3, E=E) for _ in range(2))
    inbox = TransitionInbox(rp, lanes, slots=2, slot_transitions=2 * E)
    assert inbox.layout["region_bytes"] < 8 << 20
    data = [_lane_data(E, steps, shape, seed=l) for l in range(lanes)]
    order = _drive(inbox, data, np.random.RandomState(1), max_gap=4)
    assert rp.index.head_q > rp.size
    _feed_twin(twin, E, order)
    _same_as_twin(rp, twin, "1024 lanes")
    _check_against_packer(rp, E, 3, order)


def test_a_new_writer_of_a_lane_resets_its_streams():
    """Lane 0's writer closes; lane 1's stops with a step packed (lost) and slots committed (still drained).  After
    unclaim, a new writer of each lane resets its streams on its first step: the twin takes reset_streams and then
    the step."""
    shape, E, n = (4, 12), 3, 3
    rp, twin = (_shard(shape, 96, 240, n=n, E=E, age_limit=25) for _ in range(2))
    inbox = TransitionInbox(rp, 2, slots=3, slot_transitions=2 * E)
    a0, b0, a1, b1 = (_lane_data(E, 16, shape, seed=s) for s in (40, 41, 42, 43))
    lanes = _Lanes(inbox)
    lanes.open(0)
    lanes.open(1)
    for k in range(16):
        lanes.append(0, a0, k)
        if k < 15:
            lanes.append(1, b0, k)
        if k in (4, 9, 13):
            lanes.drain()
    lanes.flush(0)
    lanes.close(0)
    inbox.unclaim(0)
    assert lanes.writers[1].packer.n_steps == 1 and len(lanes.committed[1]) == 2
    dead = lanes.abandon(1)
    inbox.unclaim(1)
    lanes.open(0)
    lanes.open(1)
    for k in range(16):
        lanes.append(0, a1, k)
        lanes.append(1, b1, k)
        if k in (0, 3, 8, 12):
            lanes.drain()
    for l in (0, 1):
        lanes.flush(l)
    lanes.drain()
    assert inbox.drain() == 0
    for l in (0, 1):
        lanes.close(l)
    dead.close()
    assert sum(1 for l, _, _ in lanes.order if l == 1) == 14 + 16          # b0's packed step 14 was lost
    _feed_twin(twin, E, lanes.order)
    _same_as_twin(rp, twin, "mid-lane reset")


def test_scan_takes_at_most_max_slots_and_release_advances_by_what_it_took():
    shape, E, S = (4, 4), 2, 4
    rp = _shard(shape, 64, 160, n=3, E=E)
    inbox = TransitionInbox(rp, 2, slots=S, slot_transitions=E)
    w = TransitionWriter(inbox, lane=1, timeout=5.0)
    obs, _, act, rew, done = _lane_data(E, 6, shape, seed=3)

    def commit(k):
        w.append_vector_step(obs[k], act[k], rew[k], done[k], obs[k + 1])
        w.flush()

    def release():
        with torch.cuda.device(inbox.device):
            _lib.check(inbox.lib.a0_tx_release(inbox._h, _lib.stream_ptr(inbox.device)), "a0_tx_release")
            torch.cuda.current_stream(inbox.device).synchronize()

    for k in range(3):
        commit(k)
    idle = (0, 0, 0)
    _scan(inbox, 1, [idle, (0, 3, 1)])
    release()
    assert int(inbox.lane_words(1)[2]) == 1
    _scan(inbox, 1, [idle, (1, 3, 1)])                                       # the next slot
    release()
    _scan(inbox, 64, [idle, (2, 3, 1)])
    release()
    _scan(inbox, 64, [idle, (3, 3, 0)])
    release()                                                                # nothing taken: nothing moves
    assert [int(x) for x in inbox.lane_words(1)[1:]] == [3, 3]
    for k in range(3, 6):
        commit(k)                                                            # slots 3, 0, 1
    _scan(inbox, 2, [idle, (3, 6, 2)])
    release()
    _scan(inbox, 64, [idle, (5, 6, 1)])
    release()
    assert [int(x) for x in inbox.lane_words(1)[1:]] == [6, 6] and int(inbox.lane_words(0)[2]) == 0
    w.close()


# -------------------------------------------------------------------------------------- 4. one step per slot
def test_a_slot_of_one_vector_step_takes_a_first_step_of_new_stacks_on_every_stream():
    """The writer's first step carries the E reset stacks and 4 new frames on every stream: 8E frames, which the
    default slot_frames of a one-step slot must hold."""
    shape, E, T, n = (4, 12), 4, 30, 3
    rp, twin = (_shard(shape, 64, 120, n=n, E=E, age_limit=25) for _ in range(2))
    inbox = TransitionInbox(rp, 1, slots=2, slot_transitions=E)
    obs, n_new, act, rew, done = _lane_data(E, T, shape, seed=5)
    first = np.random.RandomState(6).randint(0, 256, obs[0].shape, dtype=np.uint8)
    data = (np.concatenate([first[None], obs]), np.concatenate([np.full((1, E), 4), n_new]),
            np.concatenate([act[:1], act]), np.concatenate([rew[:1], rew]), np.concatenate([done[:1], done]))
    assert (stack_delta(data[0][0], data[0][1]) == 4).all()
    order = _drive(inbox, [data], np.random.RandomState(7), max_gap=2)
    _feed_twin(twin, E, order)
    _same_as_twin(rp, twin, "one step per slot")
    _check_against_packer(rp, E, n, order)


def test_a_slot_that_cannot_take_every_vector_step_is_refused():
    E = 4
    rp = _shard((4, 4), 64, 200, n=3, E=E)
    with pytest.raises(ValueError, match="slot_transitions 3 "):
        TransitionInbox(rp, 1, slot_transitions=E - 1)
    with pytest.raises(ValueError, match=f"slot_frames {8 * E - 1} "):
        TransitionInbox(rp, 1, slot_transitions=E, slot_frames=8 * E - 1)
    assert TransitionInbox(rp, 1, slot_transitions=E, slot_frames=8 * E).SF == 8 * E
    assert TransitionInbox(rp, 1, slot_transitions=E).SF == 8 * E               # the default of a one-step slot
