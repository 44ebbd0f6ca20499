"""a0_ix_merge (k shard checkpoints into one index of another capacity, frame capacity or age limit) against its
specification ring_index.merge: the target index, records, leaves, frame placements, record map, stacks and tails
agree for resizes, shorter age limits, several files of different fill levels, stale records and stream maps; later
appends plan identically; bad inputs raise and leave the target untouched; reshard_assignment gives every (file,
stream) to exactly one rank.  CPU only."""
import numpy as np
import pytest

from agent0_b200.ring_index import (SLOTS, NativeRingIndex, RingIndex, apply_rec_meta, empty_records, merge, parse_index,
                                    serialize_index)
from agent0_b200.trainer import reshard_assignment


def _source(N, NF, n, age, seed, iters, S=5, id0=0, idle=None, static=False):
    """A NativeRingIndex fed random multi-stream appends, with the RECORDS its plans write, random leaves of its
    sampleable records and a TAILS entry (the last record's frames) per stream.  ``idle``: a stream that stops for
    a while and resumes (stale records); ``static``: most steps bring no new frame (static screens)."""
    rng = np.random.RandomState(seed)
    ix = NativeRingIndex(N, NF, n, age)
    slots, info = empty_records(N)
    ids = list(range(id0, id0 + S))
    ix.plan(np.zeros(0, np.int64), np.zeros((0, 8), np.int64), np.arange(4 * S), [], [], [])
    for i, sid in enumerate(ids):
        ix.set_stack(sid, np.arange(4 * i, 4 * i + 4))
    last = {}
    for it in range(iters):
        m = int(rng.randint(1, ix.max_chunk + 1))
        active = [s for s in ids if idle is None or s != idle or not (iters // 4 <= it < 3 * iters // 4)]
        stream = rng.choice(active, size=m).astype(np.int64)
        n_new = rng.choice([0, 0, 0, 0, 1] if static else [0, 1, 1, 1, 2, 4], size=m).astype(np.int64)
        fs8 = ix.resolve_shift(stream, n_new)
        p = ix.plan(stream, fs8, np.arange(int(n_new.sum())), rng.randint(0, 18, m), rng.randn(m), rng.rand(m) < 0.1)
        apply_rec_meta(slots, info, p.rec_meta)
        for t in range(m):
            last[int(stream[t])] = fs8[t].copy()
    leaves = np.where(ix.sampleable, rng.rand(N).astype(np.float32) * 3, 0).astype(np.float32)
    tails = [(sid, last[sid]) for sid in sorted(last)]
    records = np.concatenate([slots.view(np.uint8).ravel(), info.view(np.uint8).ravel()])
    return dict(native=ix, index=parse_index(ix.serialize()), slots=slots, info=info, leaves=leaves, tails=tails, records=records)


def _both(sources, N, NF, n, age, streams=None):
    spec = RingIndex(N, NF, n, age)
    want = merge(spec, sources, streams)
    nat = NativeRingIndex(N, NF, n, age)
    got = nat.merge([s["native"] for s in sources], [s["records"] for s in sources], [s["leaves"] for s in sources],
                    streams, [s["tails"] for s in sources])
    assert nat.serialize() == serialize_index(spec, want["stacks"])
    for key in ("slots", "info", "leaves", "placements", "record_map"):
        assert np.array_equal(got[key], want[key]), key
    assert got["stride_hint"] == want["stride_hint"]
    assert len(got["tails"]) == len(want["tails"])
    for a, b in zip(got["tails"], want["tails"]):
        assert a[:3] == b[:3] and np.array_equal(a[3], b[3])
    for sid, st in want["stacks"].items():
        assert np.array_equal(nat.get_stack(sid), st)
    # every final ring slot has at most one placement, inside the resident window of the target
    assert len(set(want["placements"][:, 2].tolist())) == len(want["placements"])
    return spec, nat, want


def _check_content(sources, want, spec):
    """Every kept record the target holds names, through its slots, the frames its source record names."""
    place = {int(p): (int(j), int(f)) for j, f, p in want["placements"]}
    for j, src_pos, dst in want["record_map"]:
        if dst < 0:
            continue
        six = sources[j]["index"]
        lo = max(0, six["head_fs"] - six["NF"])
        for c in range(SLOTS):
            p = int(sources[j]["slots"][src_pos, c])
            f = lo + (p - lo % six["NF"]) % six["NF"]
            assert place[int(want["slots"][dst, c])] == (j, f)
        assert np.array_equal(want["info"][dst, :3], sources[j]["info"][src_pos, :3])
        if spec.sampleable[dst]:
            assert want["leaves"][dst] == sources[j]["leaves"][src_pos]


@pytest.mark.parametrize("N2,NF2", [(256, 2400), (128, 1200), (48, 1200), (256, 300)])
def test_one_file_into_another_capacity(N2, NF2):
    src = _source(128, 1200, 3, 32, 1, 120)
    spec, _, want = _both([src], N2, NF2, 3, 32)
    _check_content([src], want, spec)
    if N2 >= 128 and NF2 >= 1200:
        assert spec.top == src["index"]["top"]


def test_shorter_age_limit_restores_static_frames():
    src = _source(200, 2000, 1, 200, 2, 150, static=True)
    spec, _, want = _both([src], 200, 2000, 1, 16)
    _check_content([src], want, spec)
    used = {(int(j), int(f)) for j, f, _ in want["placements"]}
    assert len(want["placements"]) > len(used) or spec.head_fs > len(used)      # some frames stored twice


@pytest.mark.parametrize("n", [1, 3])
@pytest.mark.parametrize("k", [2, 3, 4])
def test_several_files(n, k):
    fills = [(64, 600, 400), (128, 900, 1), (96, 700, 200), (64, 600, 8)]
    srcs = [_source(N, NF, n, 24, 10 + j, it) for j, (N, NF, it) in enumerate(fills[:k])]
    assert srcs[0]["index"]["tail_q"] > 0 and srcs[1]["index"]["tail_q"] == 0
    spec, nat, want = _both(srcs, 256, 4000, n, 24)
    _check_content(srcs, want, spec)
    assert spec.top == sum(s["index"]["top"] for s in srcs)
    # later appends plan identically on both
    stacks = {sid: st.copy() for sid, st in want["stacks"].items()}
    rng = np.random.RandomState(5)
    for it in range(60):
        m = int(rng.randint(1, nat.max_chunk + 1))
        stream = rng.choice(sorted(stacks), size=m).astype(np.int64)
        n_new = rng.choice([0, 1, 1, 4], size=m).astype(np.int64)
        a, r, d = rng.randint(0, 18, m), rng.randn(m), rng.rand(m) < 0.1
        f1 = spec.resolve_shift(stream, n_new, stacks)
        f2 = nat.resolve_shift(stream, n_new)
        assert np.array_equal(f1, f2)
        p1 = spec.plan(stream, f1, np.arange(int(n_new.sum())), a, r, d)
        p2 = nat.plan(stream, f2, np.arange(int(n_new.sum())), a, r, d)
        for x, y in zip((p1.new_frame_pos, p1.rec_meta, p1.marks), (p2.new_frame_pos, p2.rec_meta, p2.marks)):
            assert np.array_equal(x, y), it
    assert nat.serialize() == serialize_index(spec, stacks)


def test_stale_records_stay_unsampleable():
    src = _source(400, 3000, 1, 16, 3, 200, idle=2)
    six = src["index"]
    live = [q % 400 for q in range(six["tail_q"], six["head_q"])]
    stale = [p for p in live if not six["sampleable"][p]]
    assert stale, "the idle stream left no stale record"
    spec, _, want = _both([src], 400, 3000, 1, 64)
    for j, s, d in want["record_map"]:
        if d >= 0:
            assert spec.sampleable[d] == six["sampleable"][s]


def test_stream_maps_drop_and_split():
    srcs = [_source(64, 600, 3, 24, 20, 100), _source(64, 600, 3, 24, 21, 60)]
    maps = [{0: 7, 2: 3}, {1: 0, 4: 9}]
    spec, _, want = _both(srcs, 128, 1200, 3, 24, maps)
    kept = {(0, 0), (0, 2), (1, 1), (1, 4)}
    assert set(spec.streams) <= {7, 3, 0, 9}
    assert all(t[0] in (7, 3, 0, 9) for t in want["tails"])
    n_kept = 0
    for j, src in enumerate(srcs):
        own = {}
        for sid, st in src["index"]["streams"].items():
            p = st["last_pos"] if st["last_seq"] >= src["index"]["tail_q"] else -1
            pred = {int(src["info"][q % 64, 3]): q % 64 for q in range(src["index"]["tail_q"], src["index"]["head_q"])}
            while p >= 0:
                own[p] = sid
                p = pred.get(p, -1)
        n_kept += sum(1 for sid in own.values() if (j, sid) in kept)
    assert len(want["record_map"]) == n_kept
    # the default map keeps every id of file 0 and offsets file j by j * S
    _, _, want = _both(srcs, 128, 1200, 3, 24)
    assert {t[0] for t in want["tails"]} <= set(range(10))


def test_bad_merges_raise_and_leave_the_target_untouched():
    srcs = [_source(64, 600, 3, 24, 30, 50), _source(64, 600, 3, 24, 31, 50)]
    nat = NativeRingIndex(128, 1200, 3, 24)
    before = nat.serialize()
    args = ([s["native"] for s in srcs], [s["records"] for s in srcs], [s["leaves"] for s in srcs])
    with pytest.raises(RuntimeError, match="both become stream 5"):
        nat.merge(*args, streams=[{0: 5}, {1: 5}])
    assert nat.serialize() == before
    with pytest.raises(ValueError):
        merge(RingIndex(128, 1200, 3, 24), srcs, [{0: 5}, {1: 5}])
    with pytest.raises(RuntimeError, match="n_step"):
        NativeRingIndex(128, 1200, 1, 24).merge(*args)
    with pytest.raises(ValueError):
        merge(RingIndex(128, 1200, 1, 24), srcs)
    bad = srcs[0]["info"].copy()
    live = srcs[0]["index"]["tail_q"] % 64
    bad[live, 3] = bad[(live + 1) % 64, 3] if bad[live, 3] != bad[(live + 1) % 64, 3] else -1
    recs = [np.concatenate([srcs[0]["slots"].view(np.uint8).ravel(), bad.view(np.uint8).ravel()]), srcs[1]["records"]]
    with pytest.raises(RuntimeError):
        nat.merge(args[0], recs, args[2])
    assert nat.serialize() == before
    nat.merge(*args)
    with pytest.raises(RuntimeError, match="not empty"):
        nat.merge(*args)


@pytest.mark.parametrize("G,G2", [(8, 1), (8, 4), (8, 3), (4, 8), (2, 3), (1, 1)])
def test_reshard_assignment(G, G2):
    ids = [list(range(0, 4 + r)) for r in range(G)]
    plan = reshard_assignment(G, G2, ids)
    assert len(plan) == G2
    owner = {}
    for r2, parts in enumerate(plan):
        new_ids = []
        for f, m in parts:
            for old, new in m.items():
                assert (f, old) not in owner
                owner[(f, old)] = r2
                new_ids.append(new)
        assert len(new_ids) == len(set(new_ids))
    assert set(owner) == {(f, s) for f in range(G) for s in ids[f]}
    if G2 > G:
        for r2, parts in enumerate(plan):
            assert [f for f, _ in parts] == [r2 % G] and all(a == b for a, b in parts[0][1].items())
