"""Actor-side inference on the learner's GPU (SURVEY 8f items 3 and 4).

``ActorPolicy.act`` has the signature and the random-number consumption of the reference's
``Actor.act`` (agent0/deepq/agent.py:25-39): observations u8 [E,4,H,W] in, ``(actions i64[E], mean of
the per-env max q)`` out.  Mechanically: one pinned H2D copy of the observations and of the host's
draws, ``a0_u8_to_f32`` (the ``.float().div(255)`` of agent.py:27), ``model.qval`` on PyTorch (out of
scope, SURVEY section 2), ``a0_act_epsilon_greedy`` (max, arg-max, ``np.where(rand > eps, ...)``, mean), and
ONE device->host copy + sync for the E actions and the mean, where the reference syncs twice
(``qt_arg_max.cpu()`` and ``qt_max.mean().item()``).  The draws come from numpy in the reference's
order (randint, then rand), so a seeded run chooses the same actions.

``broadcast_model`` replaces shipping ``model.state_dict()`` to every actor through courier RPC on
each call (agent0/deepq/launch.py:33-36,56-61): parameters and buffers are packed into one flat
buffer and sent with a single collective broadcast (NCCL on the GPU box, gloo in the CPU tests).
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib
from .replay import NORM_RECIP


class ActorPolicy:
    def __init__(self, cfg, model, device=None, norm_mode=NORM_RECIP, rng=None, weights=None):
        """model: the learner's DeepQNet (shared, as trainer.py:42-43 shares it with the Actors).
        norm_mode: NORM_RECIP reproduces torch's CUDA ``.div(255.0)`` bit for bit, NORM_DIV the CPU one.
        rng: a numpy RandomState-like object (default: numpy's global generator, as the reference).
        weights: a weights.WeightSubscriber whose model is ``model`` (an actor with its own copy of the net, e.g. in
        another process): ``pull_weights`` refreshes it, and ``ShardActor.sample`` does so at the start of every call,
        the cadence of the reference's actor node (launch.py:56-61)."""
        if not torch.cuda.is_available():
            raise RuntimeError("agent0_b200.ActorPolicy needs a CUDA device (no CPU fallback)")
        if weights is not None and weights.model is not model:
            raise ValueError("ActorPolicy(weights=): the subscriber must write into this policy's model")
        self.cfg, self.model, self.lib = cfg, model, _lib.load()
        self.weights = weights
        dv = device if device is not None else next(model.parameters()).device
        self.device = torch.device(dv)
        if self.device.type != "cuda":
            raise RuntimeError("agent0_b200.ActorPolicy: the model must live on a CUDA device")
        self.A = int(cfg.action_dim)
        self.norm_mode = int(norm_mode)
        self.rng = rng if rng is not None else np.random
        self._key = None

    def _buffers(self, E, obs_shape):
        # keyed on the whole shape: a call with the same E and other frames needs other buffers
        key = (E,) + tuple(obs_shape)
        if key == self._key:
            return
        dev = self.device
        n = int(np.prod(obs_shape))
        assert (E * n) % 16 == 0, "observation bytes must be a multiple of 16"
        self._obs_host = torch.empty((E,) + tuple(obs_shape), dtype=torch.uint8).pin_memory()
        self._obs_dev = torch.empty_like(self._obs_host, device=dev)
        self._st = torch.empty((E,) + tuple(obs_shape), dtype=torch.float32, device=dev)
        self._draw_host = torch.empty(2 * E, dtype=torch.float64).pin_memory()     # [rand f64 | randint i64 bits]
        self._draw_dev = torch.empty(2 * E, dtype=torch.float64, device=dev)
        self._res_dev = torch.zeros(E + 1, dtype=torch.int64, device=dev)          # [actions | mean (f32 bits)]
        self._res_host = torch.empty(E + 1, dtype=torch.int64).pin_memory()
        self._scratch = torch.zeros(2, dtype=torch.float32, device=dev)
        self._key = key

    def pull_weights(self):
        """The newest complete snapshot of the learner's weights into the model (WeightSubscriber.pull): the version
        applied, or 0 when there was nothing new (or the pull was torn and left the model as it was)."""
        if self.weights is None:
            raise RuntimeError("ActorPolicy.pull_weights: construct the policy with weights=WeightSubscriber(...)")
        return self.weights.pull()

    @torch.no_grad()
    def act(self, obs, epsilon):
        """agent.py:25-39.  obs: np.uint8 [E,4,H,W] (host).  Returns (np.int64 [E], float)."""
        obs = np.ascontiguousarray(obs, dtype=np.uint8)
        E = obs.shape[0]
        self._buffers(E, obs.shape[1:])
        dev, lib = self.device, self.lib
        self._obs_host.numpy()[...] = obs
        # the reference draws randint first, then rand (agent.py:30-36)
        action_random = self.rng.randint(0, self.A, E)
        u = self.rng.rand(E)
        d = self._draw_host.numpy()
        d[:E] = u
        d[E:].view(np.int64)[...] = action_random
        with torch.cuda.device(dev):
            st = _lib.stream_ptr(dev)
            self._obs_dev.copy_(self._obs_host, non_blocking=True)
            self._draw_dev.copy_(self._draw_host, non_blocking=True)
            _lib.check(lib.a0_u8_to_f32(self._obs_dev.data_ptr(), self._st.data_ptr(), self._obs_dev.numel(),
                                        self.norm_mode, st), "a0_u8_to_f32")
            q = self.model.qval(self._st).float().contiguous()
            assert q.shape == (E, self.A)
            _lib.check(lib.a0_act_epsilon_greedy(
                q.data_ptr(), E, self.A, float(epsilon), self._draw_dev.data_ptr(),
                self._draw_dev.data_ptr() + 8 * E, self._res_dev.data_ptr(), None, self._scratch.data_ptr(),
                self._res_dev.data_ptr() + 8 * E, st), "a0_act_epsilon_greedy")
            self._res_host.copy_(self._res_dev, non_blocking=True)
            torch.cuda.current_stream(dev).synchronize()
        r = self._res_host.numpy()
        return r[:E].copy(), float(r[E:].view(np.float32)[0])


class ShardActor:
    """``Actor.sample`` (agent0/deepq/agent.py:44-90) with the shard as the sink: the env loop, the done
    rule ``(terminal | life_loss) & ~truncated`` (agent.py:57-62) and the statistics are the
    reference's; what changes is where a transition goes.  The reference keeps an n-step tracker,
    concatenates the two 4-frame stacks and lz4-compresses 56 448 bytes per transition (agent.py:64-81);
    here each 1-step transition is appended to the HBM ring as it happens (only its new frames cross
    PCIe) and K3 folds the n steps at gather time.  ``envs`` is the vector env of
    ``make_atari`` (reset() -> (obs, info); step(a) -> (obs, reward, terminal, truncated, info)).

    Warm-up entries are REJECTED, not emulated: during the first n-1 steps of its lifetime the reference
    actor's tracker holds fewer than n transitions and it still emits an entry per env and step
    (agent.py:64-73) -- (obs_0, a_0, an L-step return with L = k+1 < n, obs_{k+1}) -- which its learner
    then bootstraps with gamma**n as if n steps had passed (agent.py:183).  A ring of 1-step records
    gathered with a fixed window has no such entry: record (e, 0) becomes sampleable once its (n-1)-th
    successor exists and then equals the reference's entry of step n-1.  ``warmup_entries_skipped`` counts
    what the reference would have emitted in addition: (n-1) * num_envs per actor lifetime, out of 1e7."""

    def __init__(self, cfg, envs, policy, replay):
        assert replay.n_gather == int(cfg.learner.n_step_q), "construct the ReplayDataset with native_nstep=True"
        self.cfg, self.envs, self.policy, self.replay = cfg, envs, policy, replay
        self.obs, _ = envs.reset()
        self.steps = 0
        self.warmup_entries_skipped = 0

    def reset(self):
        self.obs, _ = self.envs.reset()

    def sample(self, epsilon):
        """Runs ``cfg.actor.sample_steps`` vector steps.  Returns (transitions appended, episode returns,
        per-step mean max-q), i.e. the reference's (data, rs, qs) with the data already in the shard.  A policy with a
        weight subscriber first pulls the learner's newest weights (launch.py:56-61).  A sink with ``flush`` (an
        inbox.TransitionWriter in an actor process) is flushed at the end, so the call's steps reach the learner."""
        cfg = self.cfg
        if getattr(self.policy, "weights", None) is not None:
            self.policy.pull_weights()
        rs, qs, count = [], [], 0
        for _ in range(cfg.actor.sample_steps):
            if cfg.learner.noisy_net and self.steps % cfg.learner.reset_noise_freq == 0:
                self.policy.model.reset_noise()
            action, qt_max = self.policy.act(self.obs, epsilon)
            obs_next, reward, terminal, truncated, info = self.envs.step(action)
            self.steps += 1
            done = np.logical_or(terminal, info["life_loss"]) if "life_loss" in info else terminal
            done = np.logical_and(done, np.logical_not(truncated))
            self.replay.append_vector_step(np.asarray(self.obs), action, reward, done, np.asarray(obs_next))
            if self.steps < int(cfg.learner.n_step_q):      # the reference's tracker is still shorter than n here
                self.warmup_entries_skipped += len(action)
            count += len(action)
            self.obs = obs_next
            qs.append(qt_max)
            if "final_info" in info:
                for stat in info["final_info"][info["_final_info"]]:
                    rs.append(stat["episode"]["r"][0])
        if getattr(self.replay, "flush", None) is not None:      # a TransitionWriter sink commits the call's steps
            self.replay.flush()
        return count, rs, qs

    def close(self):
        self.envs.close()


def flat_state(model):
    """Parameters and buffers of ``model`` in state_dict order (what launch.py ships to the actors)."""
    return [t for t in model.state_dict().values() if torch.is_tensor(t)]


def broadcast_model(model, src=0, process_group=None):
    """One collective instead of a pickled state_dict per actor call (launch.py:33-36): pack every
    floating-point state tensor into one flat buffer, broadcast it from ``src``, unpack in place.
    Integer buffers (none in the deepq nets) are broadcast one by one.  Returns the bytes sent."""
    import torch.distributed as dist
    tensors = flat_state(model)
    if process_group is None and not dist.is_initialized():
        return 0
    fl = [t for t in tensors if t.is_floating_point()]
    sent = 0
    if fl:
        flat = torch.cat([t.detach().reshape(-1).float() for t in fl])
        dist.broadcast(flat, src=src, group=process_group)
        off = 0
        for t in fl:
            n = t.numel()
            t.detach().copy_(flat[off:off + n].view_as(t))
            off += n
        sent += flat.numel() * 4
    for t in tensors:
        if not t.is_floating_point():
            dist.broadcast(t, src=src, group=process_group)
            sent += t.numel() * t.element_size()
    return sent
