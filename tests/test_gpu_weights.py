"""K8 on the B200: weight snapshots published by the learner and pulled by actors (agent0_b200/weights.py,
csrc/a0_weights.cu).  Bit-exact round trips of every learner's state, segment tables of every shape and alignment, a
torn fetch that must leave the actor's weights alone, the publish as a node of the Trainer's captured graph, an actor
policy fed by a subscriber, subscribers in another process (same GPU, and a peer GPU when there are two), and handles of
a publisher and of a transition inbox each refused by the other kind's open."""
import multiprocessing as mp
import pickle
import time

import numpy as np
import pytest
import torch

from agent0_b200.config import make_config
from agent0_b200.weights import WeightPublisher, WeightSubscriber

pytestmark = pytest.mark.gpu

ALGOS = ["dqn", "mdqn", "c51", "qr", "iqn", "fqf"]


class _State:
    """A bare state: what WeightPublisher / WeightSubscriber read from a model is its state_dict()."""

    def __init__(self, tensors):
        self.tensors = dict(tensors)

    def state_dict(self):
        return self.tensors


def _state(model):
    return [t for t in model.state_dict().values()]


def _bits_equal(a, b):
    return all(x.shape == y.shape and torch.equal(x.contiguous().view(torch.int32), y.contiguous().view(torch.int32))
               for x, y in zip(_state(a), _state(b)))


def _perturb(model, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    with torch.no_grad():
        for t in _state(model):
            t.add_(torch.randn(t.shape, device=t.device, generator=g) * 1e-3)


@pytest.mark.parametrize("variant", ["dueling", "noisy", "channels_last"])
@pytest.mark.parametrize("algo", ALGOS)
def test_round_trip_is_bit_exact_for_every_learner(algo, variant):
    from agent0_b200.learner import make_learner
    from agent0_b200.model import DeepQNet
    kw = dict(noisy_net=True) if variant == "noisy" else {}
    cfg = make_config(algo, per=True, n_step=3, batch_size=32, dueling=True, replay_size=256, **kw)
    torch.manual_seed(1)
    learner = make_learner(cfg, device=torch.device("cuda", 0), channels_last=variant == "channels_last")
    torch.manual_seed(2)
    actor = DeepQNet(cfg).cuda()
    if variant == "channels_last":
        actor = actor.to(memory_format=torch.channels_last)
    assert not _bits_equal(actor, learner.model)
    pub = WeightPublisher(learner.model)
    sub = WeightSubscriber(pub, actor)
    assert sub.pull() == 0                                        # nothing published yet
    for v in (1, 2, 3):
        _perturb(learner.model, v)
        pub.publish()
        assert sub.pull() == v
        assert _bits_equal(actor, learner.model), f"version {v} differs"
        assert sub.pull() == 0                                    # nothing new
    h = pub.handle()
    assert pickle.loads(pickle.dumps(h)) == h and len(h["ipc"]) == 64 and h["n_words"] == sum(t.numel() for t in _state(actor))


def _segments(sizes, shift, seed):
    """Views of one storage at word offsets shift, shift + 1 + ..., so that starts fall at every 4-byte offset mod 16;
    random bit patterns (NaNs and denormals included)."""
    total = sum(sizes) + 8 * len(sizes) + 8
    g = torch.Generator(device="cuda").manual_seed(seed)
    store = torch.randint(-2**31, 2**31 - 1, (total,), dtype=torch.int32, device="cuda", generator=g).view(torch.float32)
    out, off = {}, shift
    for k, n in enumerate(sizes):
        out[f"s{k}"] = store[off:off + n]
        off += n + 1 + (k % 3)
    return out, store


@pytest.mark.parametrize("shift", [0, 1, 2, 3])
@pytest.mark.parametrize("table", ["small", "fc", "many"])
def test_segment_shapes_and_alignments(table, shift):
    rng = np.random.RandomState(shift)
    sizes = {"small": [1, 3, 31, 33, 1, 64, 5], "fc": [31, 3136 * 512, 3, 512, 33],
             "many": list(rng.randint(1, 40, 3000))}[table]
    src_t, _ = _segments(sizes, shift, 10 + shift)
    dst_t, _ = _segments(sizes, (shift + 1) % 4, 20 + shift)       # the subscriber's segments sit elsewhere mod 16
    pub = WeightPublisher(_State(src_t))
    sub = WeightSubscriber(pub, _State(dst_t))
    for v in (1, 2, 3):
        with torch.no_grad():
            for t in src_t.values():
                t.copy_(torch.randint(-2**31, 2**31 - 1, t.shape, dtype=torch.int32, device="cuda").view(torch.float32))
        pub.publish()
        assert sub.pull() == v
        for k in src_t:
            assert torch.equal(src_t[k].view(torch.int32), dst_t[k].view(torch.int32)), (k, v)


def test_torn_fetch_leaves_the_weights_and_applies_the_next_version():
    from agent0_b200.model import DeepQNet
    cfg = make_config("c51", dueling=True)
    torch.manual_seed(1)
    learner = DeepQNet(cfg).cuda()
    torch.manual_seed(2)
    actor = DeepQNet(cfg).cuda()
    pub = WeightPublisher(learner)
    sub = WeightSubscriber(pub, actor)
    ctl = pub.control_words()
    assert int(ctl[0]) & 0xFFFFFFFF == 0x57304130 and int(ctl[1]) & (2**64 - 1) == pub.hash
    assert int(ctl[2]) == pub.n_words and int(ctl[3]) == 0
    for v in (1, 2):
        _perturb(learner, v)
        pub.publish()
        assert sub.pull() == v
    before = [t.clone() for t in _state(actor)]
    _perturb(learner, 3)
    pub.publish()
    torch.cuda.synchronize()
    assert int(ctl[3]) == 3 and int(ctl[5]) == 6                   # latest = 3 in buffer 1, seq[1] = 2 * 3
    ctl[5] = 5                                                      # a writer is in buffer 1 again (protocol state)
    for _ in range(3):
        assert sub.pull() == 0                                     # torn: nothing applied
        assert all(torch.equal(a.view(torch.int32), b.view(torch.int32)) for a, b in zip(before, _state(actor)))
    st = sub.pull_async()
    torch.cuda.synchronize()
    assert int(st[0]) == 0
    _perturb(learner, 4)
    pub.publish()                                                  # version 4 goes to buffer 0
    assert sub.pull() == 4 and _bits_equal(actor, learner)
    pub.publish()                                                  # version 5 reopens and closes buffer 1
    st = sub.pull_async()
    torch.cuda.synchronize()
    assert int(st[0]) == 5 and _bits_equal(actor, learner)


def test_captured_trainer_publishes_every_step():
    from agent0_b200.model import DeepQNet
    from agent0_b200.synth import fill_shard_synthetic
    from agent0_b200.trainer import Trainer
    B, L = 32, 4
    cfg = make_config("c51", per=True, n_step=3, batch_size=B, double_q=True, dueling=True, replay_size=4096, num_envs=8)
    cfg.learner.learner_steps = L
    cfg.learner.target_update_freq = 8
    torch.manual_seed(3)
    tr = Trainer(cfg, native_nstep=True, graph=True, fused_input=True, sampler_seed=7, publish_weights=True)
    fill_shard_synthetic(tr.replay, 4096, 8, 20)
    h = tr.weight_handle()
    assert pickle.loads(pickle.dumps(h)) == h
    torch.manual_seed(4)
    actor = DeepQNet(cfg).cuda()
    sub = WeightSubscriber(tr.publisher, actor)
    for step in range(1, 5):                                       # step 1 runs eagerly and captures, 2..4 replay
        tr.learn()
        assert sub.pull() == step
        assert _bits_equal(actor, tr.learner.model), f"step {step}"
    assert tr._graphed.graph is not None
    # the default Trainer publishes nothing
    assert Trainer(cfg, native_nstep=True).publisher is None


def test_actor_policy_with_a_subscriber_acts_like_the_learners_policy():
    from agent0_b200.actor import ActorPolicy
    from agent0_b200.learner import make_learner
    from agent0_b200.model import DeepQNet
    cfg = make_config("c51", per=True, n_step=3, batch_size=32, double_q=True, dueling=True, replay_size=256, num_envs=16)
    torch.manual_seed(1)
    learner = make_learner(cfg, device=torch.device("cuda", 0))
    _perturb(learner.model, 9)
    torch.manual_seed(2)
    actor_net = DeepQNet(cfg).cuda()
    pub = WeightPublisher(learner.model)
    sub = WeightSubscriber(pub, actor_net)
    pol = ActorPolicy(cfg, actor_net, rng=np.random.RandomState(5), weights=sub)
    ref = ActorPolicy(cfg, learner.model, rng=np.random.RandomState(5))
    pub.publish()
    assert pol.pull_weights() == 1
    obs = np.random.RandomState(3).randint(0, 256, (16, 4, 84, 84)).astype(np.uint8)
    for eps in (0.0, 0.3, 0.05):
        a, m = pol.act(obs, eps)
        a_ref, m_ref = ref.act(obs, eps)
        assert np.array_equal(a, a_ref) and m == m_ref
    with pytest.raises(ValueError):
        ActorPolicy(cfg, learner.model, weights=sub)


# ---- another process ---------------------------------------------------------------------------------------------
SHAPES = [(1_000_003,), (512, 77), (3,)]


def _value(k):
    return float(np.float32(k * 0.5 + 0.25))


def _child(handle, device, n_last, ready, results, deadline_s):
    """Opens the handle on `device`, signals `ready`, pulls until it has applied version n_last or the deadline passes,
    and checks every applied snapshot: uniform, the value of its version, versions increasing."""
    out = dict(seen=[], error=None, ipc_refused=None, zero_pulls=0)
    try:
        import torch
        from agent0_b200.weights import WeightSubscriber
        torch.cuda.set_device(device)
        state = _State({f"t{i}": torch.zeros(s, device=f"cuda:{device}") for i, s in enumerate(SHAPES)})
        try:
            sub = WeightSubscriber(handle, state)
        except RuntimeError as e:
            if "cudaIpcOpenMemHandle" in str(e):
                out["ipc_refused"] = str(e)
                return
            raise
        ready.set()
        end = time.monotonic() + deadline_s
        last = 0
        while time.monotonic() < end:
            v = sub.pull()
            if v:
                vals = torch.cat([t.reshape(-1) for t in state.tensors.values()])
                want = _value(v)
                if not bool((vals == want).all()):
                    out["error"] = f"version {v}: snapshot is not uniform {want} (min {vals.min().item()}, max {vals.max().item()})"
                    return
                if v <= last:
                    out["error"] = f"version {v} after {last}"
                    return
                out["seen"].append(v)
                last = v
                if v == n_last:
                    break
            else:
                out["zero_pulls"] += 1
        sub.close()
    except Exception as e:                                          # reported, never raised past the queue
        out["error"] = repr(e)
    finally:
        ready.set()
        try:
            results.put(out, timeout=10)
        except Exception:
            pass


def _stop(p):
    if p.is_alive():
        p.terminate()
        p.join(timeout=10)
    if p.is_alive():
        p.kill()
        p.join(timeout=10)


def _cross_process(device):
    N = 200
    state = _State({f"t{i}": torch.zeros(s, device="cuda:0") for i, s in enumerate(SHAPES)})
    pub = WeightPublisher(state)
    ctx = mp.get_context("spawn")
    results, ready = ctx.Queue(), ctx.Event()
    p = ctx.Process(target=_child, args=(pub.handle(), device, N, ready, results, 60.0), daemon=True)
    p.start()
    try:
        assert ready.wait(timeout=120), "the subscriber process did not start"
        for k in range(1, N + 1):
            with torch.no_grad():
                for t in state.tensors.values():
                    t.fill_(_value(k))
            pub.publish()
            if k <= N // 2:                                        # first half paced, second half back to back
                torch.cuda.synchronize()
                time.sleep(0.002)
            if not p.is_alive():
                break
        torch.cuda.synchronize()
        out = results.get(timeout=90)
        p.join(timeout=30)
    finally:
        _stop(p)
    assert not p.is_alive()
    if out["ipc_refused"]:
        pytest.skip(f"this machine refuses to map another process's CUDA IPC handle: {out['ipc_refused']}")
    assert out["error"] is None, out["error"]
    assert out["seen"] and out["seen"][-1] == N, out["seen"][-5:]
    return out["seen"]


def test_cross_process_subscriber_on_the_same_gpu():
    seen = _cross_process(0)
    assert len(seen) >= 2


def test_cross_process_subscriber_on_a_peer_gpu():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    seen = _cross_process(1)
    assert len(seen) >= 2


def _cross_kind_child(weights_handle, inbox_handle, results):
    """Opens the inbox's handle with the publisher's region in it as a TransitionWriter, and the inbox's region as a
    WeightSubscriber whose model passes the Python-side layout check: the region's control block must refuse both."""
    out = dict(error=None, ipc_refused=None, writer=None, subscriber=None)
    try:
        import torch
        from agent0_b200.inbox import TransitionWriter
        from agent0_b200.weights import WeightSubscriber, layout_hash
        torch.cuda.set_device(0)
        state = _State({"t0": torch.zeros(1000, device="cuda:0")})
        opens = dict(
            writer=lambda: TransitionWriter(dict(inbox_handle, ipc=weights_handle["ipc"]), device=torch.device("cuda", 0)),
            subscriber=lambda: WeightSubscriber(dict(ipc=inbox_handle["ipc"], n_words=1000, layout_hash=layout_hash(state),
                                                     pci_bus_id=inbox_handle["pci_bus_id"]), state))
        for kind, open_ in opens.items():
            try:
                open_().close()
                out[kind] = "opened"
            except RuntimeError as e:
                if "cudaIpcOpenMemHandle" in str(e):
                    out["ipc_refused"] = str(e)
                    return
                out[kind] = str(e)
    except Exception as e:                                          # reported, never raised past the queue
        out["error"] = repr(e)
    finally:
        try:
            results.put(out, timeout=10)
        except Exception:
            pass


def test_a_handle_of_the_other_kind_is_refused_in_another_process():
    from agent0_b200.inbox import TransitionInbox
    from agent0_b200.replay import ReplayDataset
    cfg = make_config("c51", per=True, n_step=3, batch_size=32, replay_size=2048, num_envs=16)
    inbox = TransitionInbox(ReplayDataset(cfg, native_nstep=True), 1, slots=2)
    pub = WeightPublisher(_State({"t0": torch.zeros(1000, device="cuda:0")}))
    ctx = mp.get_context("spawn")
    results = ctx.Queue()
    p = ctx.Process(target=_cross_kind_child, args=(pub.handle(), inbox.handle(0), results), daemon=True)
    p.start()
    try:
        out = results.get(timeout=180)
        p.join(timeout=30)
    finally:
        _stop(p)
    assert not p.is_alive()
    if out["ipc_refused"]:
        pytest.skip(f"this machine refuses to map another process's CUDA IPC handle: {out['ipc_refused']}")
    assert out["error"] is None, out["error"]
    assert "is not a transition inbox's region" in out["writer"], out["writer"]
    assert "is not a weight publisher's region" in out["subscriber"], out["subscriber"]
