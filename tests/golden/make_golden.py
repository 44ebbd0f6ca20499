"""Generate the golden fixtures in this directory from the UNMODIFIED reference.

Run in the build container only (needs /root/reference, which does not exist on
the GPU box):  python tests/golden/make_golden.py

The reference tree is imported read-only with three sys.modules stubs (lz4,
prefetch_generator, atari_wrappers.make_atari); nothing in it is patched except
*instance* attributes (a scripted ``act`` on the Actor instance, a CPU data
fetcher on the Trainer instance, table-lookup networks on learner instances) so
that kernel inputs are exactly controlled.  Every array written here is an
output of reference code: agent0/deepq/{agent,replay,trainer}.py.

Fixtures:
  replay_n{1,3}.npz   Actor.sample n-step packing -> ReplayDataset entries
  per_state.npz       ReplayDataset.extend / update_priority bookkeeping
  trainer_step.npz    the real Trainer.step inner loop (IS weights, priorities)
  loss_<algo>_<dq>.npz  train_step inputs/outputs/autograd grads, six algos
  static_fns.npz      huber_qr_loss / log_softmax_stable known answers
  act.npz             Actor.act epsilon-greedy selection (python tests/golden/make_golden.py --only act)
  model_parity.npz    DeepQNet per algo x {plain, dueling, dueling+noisy}: tests/model_record.py's record
                      (python tests/golden/make_golden.py --only model_parity)
"""
import os
import sys
import tempfile
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, REPO)
sys.path.insert(0, "/root/reference")


def _stub(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


_lz4 = _stub("lz4")
_lz4.block = _stub("lz4.block", compress=lambda b: bytes(b), decompress=lambda b: b)
_stub("prefetch_generator", BackgroundGenerator=lambda it, max_prefetch=3: it)

from agent0_b200.synth import record_stream  # noqa: E402

_CURRENT_ENV = {}


class ScriptedVecEnv:
    """Replays a pre-recorded stream through the vector-env contract."""

    def __init__(self, stream):
        self.s = stream
        self.k = 0
        E = stream["obs"].shape[1]
        self.observation_space = types.SimpleNamespace(shape=stream["obs"].shape[1:])
        self.action_space = [types.SimpleNamespace(n=4)] * E

    def reset(self):
        return self.s["obs"][0].copy(), {}

    def step(self, action):
        k = self.k
        assert np.array_equal(action, self.s["action"][k])
        self.k += 1
        info = {"life_loss": self.s["life_loss"][k]}
        return (self.s["obs"][k + 1].copy(), self.s["reward"][k].copy(),
                self.s["terminal"][k].copy(), self.s["truncated"][k].copy(), info)

    def close(self):
        pass


_stub("agent0.common.atari_wrappers",
      make_atari=lambda env_id, n, **k: ScriptedVecEnv(_CURRENT_ENV["stream"]))

import agent0.deepq.agent as agents  # noqa: E402
import agent0.deepq.trainer as ref_trainer  # noqa: E402
from agent0.deepq.config import (AlgoEnum, DeviceEnum, ExpConfig,  # noqa: E402
                                 ReplayEnum)
from agent0.deepq.replay import ReplayDataset  # noqa: E402
from torch.utils.data import default_collate  # noqa: E402


def base_cfg(E=3, n=1, algo="dqn", per=False, B=8, size=256, double=False, dueling=False,
             steps=40):
    cfg = ExpConfig()
    cfg.device = DeviceEnum.cpu
    cfg.obs_shape = (4, 84, 84)
    cfg.action_dim = 4
    cfg.wandb = False
    cfg.tb = False
    cfg.logdir = tempfile.mkdtemp()
    cfg.actor.num_envs = E
    cfg.actor.sample_steps = steps
    cfg.learner.algo = AlgoEnum[algo]
    cfg.learner.n_step_q = n
    cfg.learner.batch_size = B
    cfg.learner.double_q = double
    cfg.learner.dueling_head = dueling
    cfg.replay.size = size
    cfg.replay.policy = ReplayEnum.prioritize if per else ReplayEnum.uniform
    return cfg


def scripted_actor(cfg, stream):
    _CURRENT_ENV["stream"] = stream
    actor = agents.Actor(cfg, model=torch.nn.Identity())
    script = iter(stream["action"])
    actor.act = lambda eps: (next(script), 0.0)  # instance attribute, reference untouched
    return actor


# ----------------------------------------------------------------------------- replay
def gen_replay(n):
    E, T = 3, 40
    stream = record_stream(E, T, seed=100 + n, p_terminal=0.07, p_life_loss=0.08,
                           p_truncated=0.05)
    cfg = base_cfg(E=E, n=n, steps=T)
    actor = scripted_actor(cfg, stream)
    data, _, _ = actor.sample(1.0)
    replay = ReplayDataset(cfg)
    replay.extend(data)
    items = [replay[i] for i in range(len(replay))]
    frames = np.stack([it[0] for it in items])
    out = dict(
        n_step=n, num_envs=E, steps=T, seed=100 + n, discount=cfg.learner.discount,
        stream_obs=stream["obs"], stream_action=stream["action"], stream_reward=stream["reward"],
        stream_terminal=stream["terminal"], stream_truncated=stream["truncated"],
        stream_life_loss=stream["life_loss"],
        entry_frames=frames,
        entry_action=np.array([it[1] for it in items], dtype=np.int64),
        entry_reward=np.array([it[2] for it in items], dtype=np.float64),
        entry_done=np.array([it[3] for it in items], dtype=np.bool_),
        entry_idx=np.array([it[5] for it in items], dtype=np.int64),
    )
    np.savez_compressed(os.path.join(HERE, f"replay_n{n}.npz"), **out)
    print(f"replay_n{n}: {frames.shape[0]} entries, done rate {out['entry_done'].mean():.2f}")


# ----------------------------------------------------------------------------- PER bookkeeping
def gen_per_state():
    cfg = base_cfg(per=True, size=48)
    cfg.trainer.total_steps = 400
    replay = ReplayDataset(cfg)
    rng = np.random.RandomState(7)
    dummy = (b"x", np.int64(0), np.float64(0.0), np.bool_(False))
    log = dict(op=[], count=[], ids=[], loss=[], priority=[], top=[], beta=[], max_p=[])
    for it in range(9):
        k = int(rng.randint(3, 12))
        replay.extend([dummy] * k)
        log["op"].append(0); log["count"].append(k)
        log["ids"].append(np.zeros(6, np.int64)); log["loss"].append(np.zeros(6, np.float32))
        log["priority"].append(replay.priority.numpy().copy()); log["top"].append(replay.top)
        log["beta"].append(replay.beta); log["max_p"].append(replay.max_p)
        ids = torch.from_numpy(rng.randint(0, replay.top, size=6).astype(np.int64))
        loss = torch.from_numpy((np.abs(rng.randn(6)) * (1 + it)).astype(np.float32))
        replay.update_priority(ids, loss)
        log["op"].append(1); log["count"].append(0)
        log["ids"].append(ids.numpy()); log["loss"].append(loss.numpy())
        log["priority"].append(replay.priority.numpy().copy()); log["top"].append(replay.top)
        log["beta"].append(replay.beta); log["max_p"].append(replay.max_p)
    np.savez_compressed(
        os.path.join(HERE, "per_state.npz"), size=48, alpha=cfg.replay.alpha, eps=cfg.replay.eps,
        beta0=cfg.replay.beta0, total_steps=cfg.trainer.total_steps,
        **{k: np.array(v) for k, v in log.items()})
    print("per_state: ops", len(log["op"]))


# ----------------------------------------------------------------------------- Trainer.step
class ListFetcher:
    """CPU stand-in for DataLoaderX+DataPrefetcher: same collate, scripted indices."""

    def __init__(self, replay, batches):
        self.replay, self.batches = replay, iter(batches)

    def next(self):
        return default_collate([self.replay[int(i)] for i in next(self.batches)])


def gen_trainer_step():
    E, T, n, B = 3, 30, 3, 8
    stream = record_stream(E, T, seed=321, p_terminal=0.05, p_life_loss=0.05, p_truncated=0.03)
    cfg = base_cfg(E=E, n=n, algo="c51", per=True, B=B, size=64, double=True, dueling=True, steps=T)
    cfg.trainer.training_start_steps = 10
    cfg.trainer.total_steps = 1000
    cfg.learner.learner_steps = 3
    _CURRENT_ENV["stream"] = stream
    torch.manual_seed(5)
    trainer = ref_trainer.Trainer(cfg, use_lp=True)
    actor = scripted_actor(cfg, stream)
    data, _, _ = actor.sample(1.0)
    rng = np.random.RandomState(11)
    batches = [rng.randint(0, 64, size=B) for _ in range(cfg.learner.learner_steps)]
    trainer.data_fetcher = ListFetcher(trainer.replay, batches)
    rec = dict(weights=[], q_loss=[], indices=[], batch_prio=[], rewards=[], dones=[],
               actions=[], prio_after=[], max_p_after=[], frames_crc=[])
    real_train = trainer.learner.train
    real_update = trainer.replay.update_priority

    def train_spy(d):
        frames, actions, rewards, terminals, weights, indices = d
        rec["weights"].append(weights.numpy().copy()); rec["rewards"].append(rewards.numpy().copy())
        rec["dones"].append(terminals.numpy().copy()); rec["actions"].append(actions.numpy().copy())
        rec["frames_crc"].append(frames.to(torch.uint8).numpy().astype(np.uint64).sum(axis=1))
        res = real_train(d)
        rec["q_loss"].append(res["q_loss"].numpy().copy()); rec["indices"].append(res["indices"].numpy().copy())
        return res

    def update_spy(ids, priorities):
        real_update(ids, priorities)
        rec["prio_after"].append(trainer.replay.priority.numpy().copy())
        rec["max_p_after"].append(trainer.replay.max_p)

    trainer.learner.train = train_spy
    trainer.replay.update_priority = update_spy
    trainer.step(data, [], [])
    np.savez_compressed(
        os.path.join(HERE, "trainer_step.npz"), size=64, batch=B, n_step=n, num_envs=E, steps=T,
        seed=321, top=trainer.replay.top, beta_used=cfg.replay.beta0,
        beta_after=trainer.replay.beta, alpha=cfg.replay.alpha, eps=cfg.replay.eps,
        prio_before=np.concatenate([np.ones(64 - len(data)),
                                    np.ones(len(data))]).astype(np.float32)
        if len(data) <= 64 else np.ones(64, np.float32),
        batches=np.array(batches), **{k: np.array(v) for k, v in rec.items()})
    print("trainer_step: top", trainer.replay.top, "q_loss", rec["q_loss"][0][:3])


# ----------------------------------------------------------------------------- losses
OBS_TAG, NEXT_TAG = 0.0, 1.0


def _tag(x):
    return "next" if float(x.reshape(-1)[0]) > 0.5 else "cur"


class TableNet:
    """Network stub for dqn/mdqn/c51/qr: returns pre-baked outputs keyed by input tag."""

    def __init__(self, out, qval, head):
        self.out, self._qval, self.head = out, qval, head

    def __call__(self, x):
        return self.out[_tag(x)]

    def qval(self, x):
        return self._qval[_tag(x)]


def gen_loss_simple(algo, double, B=8, A=4, seed=0):
    cfg = base_cfg(algo=algo, B=B, n=3, double=double)
    cfg.action_dim = A
    learner = getattr(agents, f"{algo.upper()}Learner")(cfg)
    g = torch.Generator().manual_seed(1000 + seed)
    N = {"dqn": 0, "mdqn": 0, "c51": cfg.learner.c51.num_atoms, "qr": cfg.learner.qr.num_atoms}[algo]
    shape = (B, A) if N == 0 else (B, A, N)
    scale = 3.0
    online_cur = (torch.randn(shape, generator=g) * scale).requires_grad_(True)
    tgt_next = torch.randn(shape, generator=g) * scale
    tgt_cur = torch.randn(shape, generator=g) * scale
    qval_next = torch.randn(B, A, generator=g) * scale          # stands in for model.qval(next_obs)
    head = learner.model.head
    learner.model = TableNet({"cur": online_cur}, {"next": qval_next}, head)
    learner.model_target = TableNet({"next": tgt_next, "cur": tgt_cur}, {}, head)
    actions = torch.randint(0, A, (B,), generator=g)
    rewards = torch.tensor(np.random.RandomState(seed).choice([-2.5, -1.0, 0.0, 1.0, 1.75, 30.0], B),
                           dtype=torch.float32)
    terminals = (torch.rand(B, generator=g) < 0.3).float()
    weights = torch.rand(B, generator=g) + 0.1
    obs = torch.full((B, 1), OBS_TAG); next_obs = torch.full((B, 1), NEXT_TAG)
    loss = learner.train_step(obs, actions, rewards, terminals, next_obs)
    loss.mul(weights).sum().backward()
    out = dict(algo=algo, double_q=double, discount=cfg.learner.discount, n_step=3,
               online_cur=online_cur.detach().numpy(), tgt_next=tgt_next.numpy(),
               tgt_cur=tgt_cur.numpy(), qval_next=qval_next.numpy(), actions=actions.numpy(),
               rewards=rewards.numpy(), terminals=terminals.numpy(), weights=weights.numpy(),
               loss=loss.detach().numpy(), grad=online_cur.grad.numpy())
    if algo == "c51":
        out.update(vmin=cfg.learner.c51.vmin, vmax=cfg.learner.c51.vmax, num_atoms=N,
                   atoms=head.atoms.reshape(-1).numpy(), delta=head.delta)
    if algo == "mdqn":
        out.update(tau=cfg.learner.mdqn.tau, lo=cfg.learner.mdqn.lo)
    np.savez_compressed(os.path.join(HERE, f"loss_{algo}_{'double' if double else 'single'}.npz"), **out)
    print(f"loss_{algo} double={double}: loss[:3]={out['loss'][:3]}")


class IQNHeadStub:
    """Stands in for model.head of iqn/fqf learners; replays pre-baked tensors in the
    order the reference's train_step asks for them (agent0/deepq/agent.py:297-388)."""

    def __init__(self, script, qval_out, prop=None):
        self.script, self.qval_out, self.prop = list(script), qval_out, prop
        self.calls = []

    def __call__(self, x, n=None, taus=None):
        q, t = self.script.pop(0)
        self.calls.append((n, None if taus is None else tuple(taus.shape)))
        return q, (taus if t is None else t)

    def qval(self, x, n=None):
        return self.qval_out

    def prop_taus(self, x):
        return self.prop


class IQNNetStub:
    def __init__(self, head):
        self.head = head

    def encoder(self, x):
        return x


def gen_loss_iqn(double, B=8, A=4, seed=0):
    cfg = base_cfg(algo="iqn", B=B, n=3, double=double)
    cfg.action_dim = A
    learner = agents.IQNLearner(cfg)
    c = cfg.learner.iqn
    g = torch.Generator().manual_seed(2000 + seed)
    q_next = torch.randn(B, c.N_dash, A, generator=g) * 3
    taus_next = torch.rand(B, c.N_dash, 1, generator=g)
    q_cur = (torch.randn(B, c.N, A, generator=g) * 3).requires_grad_(True)
    taus_cur = torch.rand(B, c.N, 1, generator=g)
    qval_next = torch.randn(B, A, generator=g) * 3
    tgt_head = IQNHeadStub([(q_next, taus_next)], qval_next)
    onl_head = IQNHeadStub([(q_cur, taus_cur)], qval_next)
    learner.model = IQNNetStub(onl_head); learner.model_target = IQNNetStub(tgt_head)
    actions = torch.randint(0, A, (B,), generator=g)
    rewards = torch.randint(-1, 2, (B,), generator=g).float() * 1.5
    terminals = (torch.rand(B, generator=g) < 0.3).float()
    weights = torch.rand(B, generator=g) + 0.1
    obs = torch.zeros(B, 1); next_obs = torch.ones(B, 1)
    loss = learner.train_step(obs, actions, rewards, terminals, next_obs)
    loss.mul(weights).sum().backward()
    np.savez_compressed(
        os.path.join(HERE, f"loss_iqn_{'double' if double else 'single'}.npz"),
        algo="iqn", double_q=double, discount=cfg.learner.discount, n_step=3,
        q_cur=q_cur.detach().numpy(), taus_cur=taus_cur.numpy(), q_next=q_next.numpy(),
        qval_next=qval_next.numpy(), actions=actions.numpy(), rewards=rewards.numpy(),
        terminals=terminals.numpy(), weights=weights.numpy(), loss=loss.detach().numpy(),
        grad=q_cur.grad.numpy())
    print(f"loss_iqn double={double}: loss[:3]={loss.detach().numpy()[:3]}")


def gen_loss_fqf(double, B=8, A=4, seed=0):
    cfg = base_cfg(algo="fqf", B=B, n=3, double=double)
    cfg.action_dim = A
    learner = agents.FQFLearner(cfg)
    F_ = cfg.learner.iqn.F
    g = torch.Generator().manual_seed(3000 + seed)
    frac_logits = (torch.randn(B, F_, generator=g)).requires_grad_(True)
    probs = frac_logits.log_softmax(-1).exp()
    taus = torch.cat((torch.zeros(B, 1), torch.cumsum(probs, -1)), -1)
    taus_hat = (taus[:, :-1] + taus[:, 1:]).detach() / 2.0
    taus3, taus_hat3 = taus.unsqueeze(-1), taus_hat.unsqueeze(-1)
    q_hat = (torch.randn(B, F_, A, generator=g) * 3).requires_grad_(True)
    q_next = torch.randn(B, F_, A, generator=g) * 3
    # interior quantile values, made mostly monotone so both sign branches are exercised
    q_bar = torch.sort(torch.randn(B, F_ - 1, A, generator=g) * 3, dim=1)[0]
    q_bar = q_bar + torch.randn(B, F_ - 1, A, generator=g) * 0.5
    qval_next = torch.randn(B, A, generator=g) * 3
    onl_head = IQNHeadStub([(q_hat, None), (q_bar, None)], qval_next, prop=(taus3, taus_hat3, None))
    tgt_head = IQNHeadStub([(q_next, None)], qval_next)
    learner.model = IQNNetStub(onl_head); learner.model_target = IQNNetStub(tgt_head)
    actions = torch.randint(0, A, (B,), generator=g)
    rewards = torch.randint(-1, 2, (B,), generator=g).float()
    terminals = (torch.rand(B, generator=g) < 0.3).float()
    weights = torch.rand(B, generator=g) + 0.1
    obs = torch.zeros(B, 1); next_obs = torch.ones(B, 1)
    loss, fraction_loss = learner.train_step(obs, actions, rewards, terminals, next_obs)
    taus.retain_grad()
    fraction_loss.mul(weights).sum().backward(retain_graph=True)
    grad_taus = taus.grad.numpy().copy()
    loss.mul(weights).sum().backward()
    np.savez_compressed(
        os.path.join(HERE, f"loss_fqf_{'double' if double else 'single'}.npz"),
        algo="fqf", double_q=double, discount=cfg.learner.discount, n_step=3,
        taus=taus.detach().numpy(), taus_hat=taus_hat.numpy(), q_hat=q_hat.detach().numpy(),
        q_next=q_next.numpy(), q_bar=q_bar.numpy(), qval_next=qval_next.numpy(),
        actions=actions.numpy(), rewards=rewards.numpy(), terminals=terminals.numpy(),
        weights=weights.numpy(), loss=loss.detach().numpy(),
        fraction_loss=fraction_loss.detach().numpy(), grad=q_hat.grad.numpy(), grad_taus=grad_taus)
    print(f"loss_fqf double={double}: loss[:2]={loss.detach().numpy()[:2]} "
          f"frac[:2]={fraction_loss.detach().numpy()[:2]}")


def gen_learner(algo, double, dueling):
    """Two real BaseLearner.train() updates on CPU (real DeepQNet, Adam, target sync) from a fixed
    seed, on batches taken from replay_n3.npz.  Pins the whole learner path: frame split, the
    train_step rule, the weighted SUM backward, the optimizer step and (FQF) the fraction step."""
    g = np.load(os.path.join(HERE, "replay_n3.npz"))
    B = 8
    cfg = base_cfg(algo=algo, B=B, n=3, double=double, dueling=dueling, per=True)
    cfg.learner.target_update_freq = 2
    torch.manual_seed(4242)
    learner = getattr(agents, f"{algo.upper()}Learner")(cfg)
    rng = np.random.RandomState(17)
    out = dict(algo=algo, double_q=double, dueling=dueling, seed=4242, batch=B)
    for it in range(3):
        idx = rng.randint(0, len(g["entry_action"]), B)
        w = (rng.rand(B) + 0.1).astype(np.float32)
        data = (torch.from_numpy(g["entry_frames"][idx]).float(), torch.from_numpy(g["entry_action"][idx]).float(),
                torch.from_numpy(g["entry_reward"][idx]).float(), torch.from_numpy(g["entry_done"][idx]).float(),
                torch.from_numpy(w), torch.from_numpy(idx).float())
        res = learner.train(data)
        out[f"idx{it}"] = idx; out[f"w{it}"] = w
        out[f"q_loss{it}"] = res["q_loss"].numpy()
        if res["fraction_loss"] is not None:
            out[f"fraction_loss{it}"] = res["fraction_loss"].numpy()
    out["param_abs_sum"] = np.array([p.detach().abs().sum().item() for p in learner.model.parameters()])
    out["target_abs_sum"] = np.array([p.detach().abs().sum().item() for p in learner.model_target.parameters()])
    out["update_steps"] = learner.update_steps
    np.savez_compressed(os.path.join(HERE, f"learner_{algo}.npz"), **out)
    print(f"learner_{algo}: q_loss0[:2]={out['q_loss0'][:2]} q_loss2[:2]={out['q_loss2'][:2]}")


def gen_static_fns():
    g = torch.Generator().manual_seed(77)
    q = torch.randn(5, 1, 16, generator=g) * 2
    qt = torch.randn(5, 12, 1, generator=g) * 2
    qt[0, 0, 0] = q[0, 0, 0] + 1.0   # |u| == 1 edge of smooth_l1
    qt[1, 1, 0] = q[1, 0, 1]         # u == 0 edge of the indicator
    taus = torch.rand(5, 1, 16, generator=g)
    hq = agents.BaseLearner.huber_qr_loss(q, qt, taus)
    logits = torch.randn(6, 18, generator=g) * 4
    lss = agents.BaseLearner.log_softmax_stable(logits, 0.03)
    lss_default = agents.BaseLearner.log_softmax_stable(logits)
    np.savez_compressed(os.path.join(HERE, "static_fns.npz"), q=q.numpy(), q_target=qt.numpy(),
                        taus=taus.numpy(), huber_qr=hq.numpy(), logits=logits.numpy(),
                        lss_tau003=lss.numpy(), lss_default=lss_default.numpy())
    print("static_fns ok")


def gen_act():
    """The unmodified Actor.act (agent.py:25-39) with the real DeepQNet on CPU: per call the q-values it
    computed (captured from model.qval), numpy's seed, the chosen actions and the returned mean."""
    E, T = 16, 6
    out = {}
    for algo in ("dqn", "c51"):
        torch.manual_seed(7)
        stream = record_stream(E, T, seed=321, p_terminal=0.05, p_life_loss=0.05, p_truncated=0.02)
        cfg = base_cfg(E=E, n=1, algo=algo, steps=T, dueling=(algo == "c51"))
        _CURRENT_ENV["stream"] = stream
        actor = agents.Actor(cfg)
        seen = []
        inner = actor.model.qval
        actor.model.qval = lambda st: (seen.append((st.clone(), inner(st))), seen[-1][1])[1]   # instance attribute
        qs, sts, acts, means, epss, seeds = [], [], [], [], [], []
        for k, eps in enumerate((0.0, 0.05, 0.3, 0.7, 1.0, 0.5)):
            actor.obs = stream["obs"][k]
            np.random.seed(1000 + k)
            a, m = actor.act(eps)
            st, q = seen[-1]
            qs.append(q.numpy().copy()); sts.append(st.numpy().copy()); acts.append(np.asarray(a, dtype=np.int64))
            means.append(m); epss.append(eps); seeds.append(1000 + k)
        out.update({f"{algo}_q": np.stack(qs), f"{algo}_action": np.stack(acts), f"{algo}_qmax_mean": np.array(means, dtype=np.float64),
                    f"{algo}_st_first": sts[0], f"{algo}_obs_first": stream["obs"][0]})
        out["epsilon"], out["np_seed"] = np.array(epss), np.array(seeds)
    np.savez_compressed(os.path.join(HERE, "act.npz"), **out)
    print("act ok:", {k: v.shape for k, v in out.items()})


def gen_model_parity():
    """The reference's agent0.deepq.model.DeepQNet, recorded by tests/model_record.py (what
    tests/test_model_parity.py compares agent0_b200.model against), six algorithms x three head variants."""
    from agent0.deepq.model import DeepQNet
    from tests.model_record import ALGOS, VARIANTS, key, record
    out = {}
    for algo in ALGOS:
        for dueling, noisy in VARIANTS:
            cfg = ExpConfig()
            cfg.obs_shape, cfg.action_dim = (4, 84, 84), 6
            cfg.learner.algo, cfg.learner.dueling_head, cfg.learner.noisy_net = AlgoEnum[algo], dueling, noisy
            for k, v in record(lambda: DeepQNet(cfg), algo).items():
                out[f"{key(algo, dueling, noisy)}/{k}"] = v
    np.savez_compressed(os.path.join(HERE, "model_parity.npz"), **out)
    print(f"model_parity: {len(out)} arrays")


if __name__ == "__main__":
    np.random.seed(0)
    torch.manual_seed(0)
    if "--only" in sys.argv:
        globals()["gen_" + sys.argv[sys.argv.index("--only") + 1]]()
        sys.exit(0)
    gen_replay(1)
    gen_replay(3)
    gen_per_state()
    gen_trainer_step()
    for algo in ("dqn", "mdqn", "c51", "qr"):
        for dq in (False, True):
            if algo == "mdqn" and dq:
                continue  # MDQNLearner ignores double_q (agent0/deepq/agent.py:193-215)
            gen_loss_simple(algo, dq)
    for dq in (False, True):
        gen_loss_iqn(dq)
        gen_loss_fqf(dq)
    gen_static_fns()
    for algo, dq, du in (("dqn", True, False), ("mdqn", False, True), ("c51", True, True), ("qr", False, False),
                         ("iqn", True, True), ("fqf", True, False)):
        gen_learner(algo, dq, du)
    gen_model_parity()
