"""K9 on the B200: transitions appended by actors through the learner's inbox (agent0_b200/inbox.py,
csrc/a0_inbox.cu).  The shard a drain builds must be bit for bit the shard in-process ``append_vector_step`` calls
build in the drain order; back-pressure, uncommitted and malformed slots, lane claims, and writers in another process
(same GPU, a peer GPU when there are two, and the full actor/learner loop with weight snapshots)."""
import multiprocessing as mp
import time

import numpy as np
import pytest
import torch

from agent0_b200 import _lib
from agent0_b200.config import make_config
from agent0_b200.inbox import SlotPacker, TransitionInbox, TransitionWriter
from agent0_b200.replay import ReplayDataset
from agent0_b200.ring_index import stack_delta
from agent0_b200.synth import SyntheticStreams

pytestmark = pytest.mark.gpu

E = 16


def _cfg(replay_size=2048, sample_steps=10):
    cfg = make_config("c51", per=True, n_step=3, batch_size=32, double_q=True, dueling=True, replay_size=replay_size,
                      num_envs=E)
    cfg.actor.sample_steps = sample_steps
    return cfg


def _steps(seed, n):
    """n vector steps of one SyntheticStreams: (obs, action, reward, done, obs_next)."""
    env = SyntheticStreams(E, seed=seed, p_terminal=0.02, p_life_loss=0.03, p_truncated=0.01)
    obs, _ = env.reset()
    out = []
    for _ in range(n):
        a = env.sample_actions()
        nxt, r, term, trunc, info = env.step(a)
        done = np.logical_and(np.logical_or(term, info["life_loss"]), np.logical_not(trunc))
        out.append((obs, a, r, done, nxt))
        obs = nxt
    return out


def _reference(cfg, order):
    """An in-process shard fed ``order``: (lane, step) pairs, with append_vector_step and the lane's stream ids."""
    ref = ReplayDataset(cfg, native_nstep=True)
    for lane, (obs, a, r, d, nxt) in order:
        ref.append_vector_step(obs, a, r, d, nxt, streams=np.arange(E) + lane * E)
    return ref


def _state(rp, with_priorities=True):
    torch.cuda.synchronize()
    pos = np.flatnonzero(rp.index.sampleable)
    st = dict(frames=rp.frames.clone(), index=bytes(rp.index.serialize()), top=rp.top, beta=rp.beta, pos=pos)
    if len(pos):
        g = rp.gather(torch.as_tensor(pos, device=rp.device))
        st["records"] = [x.clone() for x in g if x is not None and torch.is_tensor(x)]
    if with_priorities:
        st["tree"], st["max_p"] = rp.tree.clone(), rp.max_p
    return st


def _assert_same(a, b, what=""):
    assert a.keys() == b.keys()
    assert a["top"] == b["top"], what
    assert a["beta"] == b["beta"], what
    assert np.array_equal(a["pos"], b["pos"]), what
    assert a["index"] == b["index"], f"{what}: serialized index differs"
    assert torch.equal(a["frames"], b["frames"]), f"{what}: frame ring differs"
    for x, y in zip(a.get("records", []), b.get("records", [])):
        assert torch.equal(x, y), f"{what}: gathered records differ"
    if "tree" in a:
        assert torch.equal(a["tree"], b["tree"]), f"{what}: tree differs"
        assert a["max_p"] == b["max_p"], what


def _run(lanes, n_steps, drains, flush_every_step=False, slots=3, steps_per_slot=5):
    """Writers on ``lanes`` lanes append n_steps vector steps each (the lanes interleaved step by step); the inbox is
    drained after the steps listed in ``drains``.  Returns the shard's state and the reference's."""
    cfg = _cfg()
    rp = ReplayDataset(cfg, native_nstep=True)
    inbox = TransitionInbox(rp, lanes, slots=slots, slot_transitions=E * steps_per_slot)
    writers = [TransitionWriter(inbox, lane=l, timeout=5.0) for l in range(lanes)]
    data = [_steps(100 + l, n_steps) for l in range(lanes)]
    done_steps = [0] * lanes            # steps in committed slots, per lane
    drained = [0] * lanes
    order = []
    total = 0

    def drain():
        nonlocal total
        got = inbox.drain()
        want = 0
        for l in range(lanes):
            order.extend((l, s) for s in data[l][drained[l]:done_steps[l]])
            want += E * (done_steps[l] - drained[l])
            drained[l] = done_steps[l]
        assert got == want
        total += got

    for k in range(n_steps):
        for l, w in enumerate(writers):
            before = w.committed
            w.append_vector_step(*data[l][k])
            if flush_every_step:
                w.flush()
            if w.committed != before or flush_every_step:
                done_steps[l] = k + 1 - w.packer.n_steps
        if k in drains:
            drain()
    for l, w in enumerate(writers):
        w.flush()
        done_steps[l] = n_steps
    drain()
    assert total == lanes * n_steps * E
    assert inbox.drain() == 0
    return _state(rp), _state(_reference(cfg, order))


def test_two_lanes_equal_the_in_process_shard_in_drain_order():
    rng = np.random.RandomState(0)
    drains, k = set(), 0
    while k < 240:
        k += int(rng.randint(1, 13))
        drains.add(k)
    got, want = _run(2, 240, drains)
    assert got["top"] > 0 and got["index"] and len(got["pos"]) > 1000
    _assert_same(got, want, "two lanes")


@pytest.mark.parametrize("schedule", ["every_step", "irregular", "rare"])
def test_one_lane_does_not_depend_on_where_the_drains_fall(schedule):
    n = 150
    if schedule == "every_step":
        got, want = _run(1, n, set(range(n)), flush_every_step=True)
    elif schedule == "irregular":
        got, want = _run(1, n, {3, 4, 15, 27, 28, 39, 50, 62, 73, 85, 96, 108, 119, 131, 142})   # gaps <= 12 steps
    else:
        got, want = _run(1, n, set(range(0, n, 14)), slots=4, steps_per_slot=4)
    _assert_same(got, want, schedule)


def test_back_pressure_reports_full_and_everything_arrives_once():
    cfg = _cfg()
    rp = ReplayDataset(cfg, native_nstep=True)
    inbox = TransitionInbox(rp, 1, slots=2, slot_transitions=E)           # one vector step per slot
    w = TransitionWriter(inbox, lane=0, timeout=0.2)
    data = _steps(7, 6)
    for s in data[:3]:
        w.append_vector_step(*s)                                             # steps 0, 1 committed, 2 packed
    assert w.committed == 2
    t0 = time.monotonic()
    with pytest.raises(TimeoutError):
        w.append_vector_step(*data[3])                                       # step 2's commit finds both slots full
    assert time.monotonic() - t0 >= 0.2
    assert int(w._status_host[0]) == _lib.TX_FULL
    assert w.committed == 2 and w.packer.n_steps == 1                        # step 3 was not taken
    assert inbox.drain() == 2 * E
    w.append_vector_step(*data[3])
    w.flush()                                                                # steps 2 and 3
    assert inbox.drain() == 2 * E
    w.append_vector_step(*data[4])
    w.append_vector_step(*data[5])
    w.flush()
    assert inbox.drain() == 2 * E
    assert inbox.drain() == 0
    _assert_same(_state(rp), _state(_reference(cfg, [(0, s) for s in data])), "back-pressure")


def _packed_slot(inbox, data, reset=True):
    L = inbox.layout
    buf = np.zeros(L["slot_bytes"], dtype=np.uint8)
    p = SlotPacker(buf, L, inbox.T, inbox.SF, inbox.F)
    for k, (obs, a, r, d, nxt) in enumerate(data):
        dk = stack_delta(obs, nxt)
        parts = ([obs.reshape(4 * E, inbox.F)] if reset and k == 0 else []) + \
            [nxt[e, 4 - dk[e]:].reshape(-1, inbox.F) for e in range(E)]
        p.add(reset and k == 0, np.arange(E), dk, a, r, d, np.concatenate(parts))
    return buf


def test_an_uncommitted_slot_is_never_ingested_and_a_committed_one_once():
    cfg = _cfg()
    rp = ReplayDataset(cfg, native_nstep=True)
    inbox = TransitionInbox(rp, 1, slots=2, slot_transitions=4 * E)
    data = _steps(9, 3)
    inbox.slot_bytes(0, 0).copy_(torch.from_numpy(_packed_slot(inbox, data)).to(rp.device))
    words = inbox.lane_words(0)
    for _ in range(3):
        assert inbox.drain() == 0                                            # written, not committed
    assert rp.top == 0 and int(words[2]) == 0
    words[1] += 1                                                            # the commit
    assert inbox.drain() == 3 * E
    assert inbox.drain() == 0
    assert int(words[1]) == int(words[2]) == 1
    _assert_same(_state(rp), _state(_reference(cfg, [(0, s) for s in data])), "partial slot")


@pytest.mark.parametrize("kind", ["n_new", "stream", "frames", "transitions"])
def test_a_malformed_slot_fails_every_drain_and_leaves_the_shard(kind):
    cfg = _cfg()
    rp = ReplayDataset(cfg, native_nstep=True)
    inbox = TransitionInbox(rp, 2, slots=2, slot_transitions=4 * E)
    good = TransitionWriter(inbox, lane=0)
    data = _steps(11, 4)
    for s in data[:2]:
        good.append_vector_step(*s)
    good.flush()
    assert inbox.drain() == 2 * E
    for s in data[2:]:
        good.append_vector_step(*s)
    good.flush()                                                             # lane 0: one good slot waiting
    buf = _packed_slot(inbox, _steps(12, 2))
    L = inbox.layout
    if kind == "n_new":
        buf[L["n_new"]:L["n_new"] + 8 * inbox.T].view(np.int64)[3] = 5
    elif kind == "stream":
        buf[L["stream"]:L["stream"] + 8 * inbox.T].view(np.int64)[0] = E
    elif kind == "frames":
        buf[16:24].view(np.int64)[0] += 1
    else:
        buf[0:8].view(np.int64)[0] = inbox.T + 1
    inbox.slot_bytes(1, 0).copy_(torch.from_numpy(buf).to(rp.device))
    inbox.lane_words(1)[1] += 1
    before = _state(rp)
    for _ in range(2):
        with pytest.raises(RuntimeError, match="lane 1, slot 0 is malformed"):
            inbox.drain()
        _assert_same(_state(rp), before, "after a failed drain")
    assert int(inbox.lane_words(0)[2]) == 1 and int(inbox.lane_words(1)[2]) == 0    # nothing released


def test_lane_claims():
    cfg = _cfg()
    rp = ReplayDataset(cfg, native_nstep=True)
    inbox = TransitionInbox(rp, 2, slots=2)
    a = TransitionWriter(inbox, lane=0)
    b = TransitionWriter(inbox, lane=1)
    with pytest.raises(RuntimeError, match="claimed by another writer"):
        TransitionWriter(inbox, lane=0)
    inbox.unclaim(0)                                                         # writer a is presumed dead
    c = TransitionWriter(inbox, lane=0)
    a.close()                                                                # a stale writer cannot free c's lane
    with pytest.raises(RuntimeError, match="claimed by another writer"):
        TransitionWriter(inbox, lane=0)
    c.close()
    d = TransitionWriter(inbox, lane=0)                                      # closing hands the lane back
    assert int(inbox.lane_words(0)[0]) != 0 and int(inbox.lane_words(1)[0]) != 0
    d.close()
    b.close()
    assert int(inbox.lane_words(0)[0]) == 0 and int(inbox.lane_words(1)[0]) == 0
    with pytest.raises(ValueError):
        TransitionWriter(inbox)


# ---- another process ---------------------------------------------------------------------------------------------
class _Scripted:
    """An actor policy with scripted actions: numpy draws from its own seed, no network."""

    def __init__(self, seed):
        self.rng = np.random.RandomState(seed)

    def act(self, obs, epsilon):
        return self.rng.randint(0, 4, len(obs)).astype(np.int64), 0.0


def _child(handle, device, calls, sample_steps, weights_handle, ready, results):
    out = dict(error=None, ipc_refused=None, count=0, versions=[])
    try:
        import torch
        from agent0_b200.actor import ActorPolicy, ShardActor
        from agent0_b200.inbox import TransitionWriter
        torch.cuda.set_device(device)
        cfg = _cfg(sample_steps=sample_steps)
        try:
            writer = TransitionWriter(handle, device=torch.device("cuda", device), timeout=60.0)
        except RuntimeError as e:
            if "cudaIpcOpenMemHandle" in str(e):
                out["ipc_refused"] = str(e)
                return
            raise
        if weights_handle is None:
            policy = _Scripted(21)
        else:
            from agent0_b200.model import DeepQNet
            from agent0_b200.weights import WeightSubscriber
            net = DeepQNet(cfg).cuda(device)
            policy = ActorPolicy(cfg, net, rng=np.random.RandomState(21), weights=WeightSubscriber(weights_handle, net))
        actor = ShardActor(cfg, SyntheticStreams(E, seed=20, p_terminal=0.02, p_life_loss=0.03, p_truncated=0.01),
                           policy, writer)
        ready.set()
        for _ in range(calls):
            n, _, qs = actor.sample(0.1)
            out["count"] += n
            if weights_handle is not None:
                out["versions"].append(policy.weights.version)
                if not all(np.isfinite(qs)):
                    out["error"] = f"non-finite q {qs}"
                    return
        writer.close()
    except Exception as e:                                                   # reported, never raised past the queue
        out["error"] = repr(e)
    finally:
        ready.set()
        try:
            results.put(out, timeout=10)
        except Exception:
            pass


def _cross_process(device, calls=12, sample_steps=10, weights=False):
    from agent0_b200.actor import ShardActor
    from agent0_b200.trainer import Trainer
    cfg = _cfg(sample_steps=sample_steps)
    cfg.learner.learner_steps = 2
    cfg.learner.target_update_freq = 4
    cfg.trainer.training_start_steps = 200
    torch.manual_seed(5)
    tr = Trainer(cfg, native_nstep=True, graph=True, fused_input=True, sampler_seed=3, inbox_lanes=1,
                 publish_weights=weights)
    ctx = mp.get_context("spawn")
    results, ready = ctx.Queue(), ctx.Event()
    p = ctx.Process(target=_child, args=(tr.inbox_handle(0), device, calls, sample_steps,
                                         tr.weight_handle() if weights else None, ready, results), daemon=True)
    p.start()
    losses, out = [], None
    try:
        assert ready.wait(timeout=180), "the actor process did not start"
        want = calls * sample_steps * E
        end = time.monotonic() + 180
        while tr.frame_count < want and time.monotonic() < end:
            stats = tr.step()
            if stats["loss"] is not None:
                losses.append(stats["loss"])
            if not p.is_alive():
                tr.step()                                                    # what the actor committed last
                break
            time.sleep(0.005)
        out = results.get(timeout=90)
        p.join(timeout=30)
    finally:
        if p.is_alive():
            p.terminate()
            p.join(timeout=10)
        if p.is_alive():
            p.kill()
            p.join(timeout=10)
    assert not p.is_alive()
    if out["ipc_refused"]:
        pytest.skip(f"this machine refuses to map another process's CUDA IPC handle: {out['ipc_refused']}")
    assert out["error"] is None, out["error"]
    assert out["count"] == calls * sample_steps * E and tr.frame_count == out["count"]
    return tr, out, losses, cfg


def _scripted_reference(cfg, calls):
    from agent0_b200.actor import ShardActor
    ref = ReplayDataset(cfg, native_nstep=True)
    actor = ShardActor(cfg, SyntheticStreams(E, seed=20, p_terminal=0.02, p_life_loss=0.03, p_truncated=0.01),
                       _Scripted(21), ref)
    for _ in range(calls):
        actor.sample(0.1)
    return ref


def _check_against_reference(tr, cfg, calls):
    ref = _scripted_reference(cfg, calls)
    # the learner's updates rewrite priorities, so the tree and max_p are not compared
    _assert_same(_state(tr.replay, with_priorities=False), _state(ref, with_priorities=False), "cross-process")


def test_another_process_on_the_same_gpu():
    tr, out, losses, cfg = _cross_process(0)
    assert tr._graphed is not None and tr._graphed.graph is not None
    assert losses and all(np.isfinite(losses))
    _check_against_reference(tr, cfg, 12)


def test_another_process_on_a_peer_gpu():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    tr, out, losses, cfg = _cross_process(1)
    _check_against_reference(tr, cfg, 12)


def test_full_loop_with_weight_snapshots():
    tr, out, losses, cfg = _cross_process(0, calls=10, weights=True)
    v = out["versions"]
    assert v == sorted(v) and v[-1] >= 1, v
    assert losses and all(np.isfinite(losses))
    assert tr.learner.update_steps > 0
