"""The hot loop of the reference's ``Trainer.step`` (agent0/deepq/trainer.py:74-119) on the
HBM-resident shard: extend -> L x {sample, IS weights, learner.train, update_priority}.

What changes mechanically: the DataLoaderX/DataPrefetcher pump (trainer.py:63-72) disappears --
one K2a launch draws all ``learner_steps`` batches and one K3 launch gathers them; IS weights come
out of the sampler's epilogue instead of ``priority.sum().item()`` over a million CPU floats
(trainer.py:91-94); nothing is copied to the host inside the loop.  Drawing the L batches up front
matches what the reference effectively does: its 2 DataLoader workers and 3-deep prefetch queue
sample several batches ahead with a fork-time snapshot of the priorities (SURVEY Q4).
"""
from __future__ import annotations

import os
from collections import deque

import numpy as np
import torch

from .learner import make_learner
from .replay import NORM_RECIP, ReplayDataset, split_batches


def _learner_data(b):
    """The reference's ``data`` tuple of BaseLearner.train (agent.py:126-131); with the fused gather the
    first field is the (obs, next_obs) f32 pair instead of the u8 frames."""
    frames = (b.obs, b.next_obs) if b.frames is None else b.frames
    return (frames, b.actions, b.rewards_f32, b.terminals_f32, b.weights, b.indices)


class GraphedUpdates:
    """The L learner updates of one Trainer.step -- CNN forward (online + target), K4, backward from
    the kernel's gradient, Adam, K2b priority write-back, L times -- as ONE CUDA graph replay over
    static batch buffers (SURVEY 8f item 2).  The draw (uniforms, K2a, K3) is part of the graph:
    ``top`` and ``beta`` are read from device memory that ``push_dynamic`` refreshes before every
    replay.  The first call runs eagerly (it is also the warm-up) and captures; later calls replay.
    At batch 32 the eager loop is bound by ~150 kernel launches per update; the replay is not."""

    def __init__(self, learner, replay, batch_size, learner_steps, normalized=None, sampler_seed=None, obs_dtype=None,
                 replacement=True, publisher=None):
        """publisher (weights.WeightPublisher, optional): publishes the model after the L updates, as the last node of
        the graph."""
        import torch
        assert learner.capturable, "construct the learner with capturable=True"
        self.publisher = publisher
        freq = learner.cfg.learner.target_update_freq
        assert freq % learner_steps == 0, "target_update_freq must be a multiple of learner_steps for graphed updates"
        self.torch, self.learner, self.replay = torch, learner, replay
        self.B, self.L = int(batch_size), int(learner_steps)
        self.normalized = normalized
        self.sampler_seed = sampler_seed
        self.obs_dtype = obs_dtype
        self.replacement = bool(replacement)
        self.static = replay.alloc_batch(self.B * self.L, normalized=normalized, obs_dtype=obs_dtype or torch.float32)
        self.graph, self.outs = None, None

    def _updates(self):
        self.replay.sample(self.B, k_batches=self.L, out=self.static, dynamic=True, normalized=self.normalized,
                           seed=self.sampler_seed, obs_dtype=self.obs_dtype, replacement=self.replacement)
        outs = []
        for b in split_batches(self.static, self.B):
            result = self.learner.update(_learner_data(b))
            self.replay.update_priority(result["indices"], result["q_loss"])
            outs.append((result["q_loss"], result["fraction_loss"]))
        if self.publisher is not None:
            self.publisher.publish()
        return outs

    def run(self):
        torch = self.torch
        self.replay.push_dynamic()
        if self.graph is None:
            outs = self._updates()                       # eager: real updates + warm-up
            steps = self.learner.update_steps
            torch.cuda.synchronize(self.replay.device)
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):           # capture only records, nothing executes
                self.outs = self._updates()
            self.learner.update_steps = steps
        else:
            self.graph.replay()
            self.learner.update_steps += self.L
            outs = self.outs
        self.learner.sync_target()
        return outs


class Trainer:
    def __init__(self, cfg, process_group=None, native_nstep=False, graph=False, fused_input=False, sampler_seed=None,
                 global_is_max=False, amp=False, channels_last=None, replacement=True, publish_weights=False, inbox_lanes=0,
                 inbox_kw=None, **replay_kw):
        """graph=True: the learner updates of a step run as one CUDA-graph replay (GraphedUpdates).
        fused_input=True: K3 writes the learner's normalised f32 obs / next_obs directly
        (a0_rb_gather_f32) instead of u8 frames that torch then casts, divides and splits
        (agent.py:129-135); ``x * fl(1/255)``, i.e. bit-identical to torch's CUDA ``.div(255)``.
        sampler_seed: the prioritized draw takes its uniforms from the sampler's own Philox generator
        (a0_pt_sample_rng) instead of torch's CUDA generator.
        native_nstep=True needs a ShardActor / append_steps feed: ``step(transitions)`` takes the reference actor's
        already n-step-folded tuples, which such a shard refuses.
        amp=True (opt-in, implies fused_input): K3 writes obs / next_obs as bf16 (a0_rb_gather_bf16) and the networks run
        under bf16 autocast with channels-last convolutions (``channels_last``, default = amp; torch converts the two
        [B,4,84,84] inputs, < 1 % of the update); parameters, Adam, K4 and the priorities stay fp32
        (BaseLearner(amp_dtype=)).  Not the reference's arithmetic, so outside the parity contract.  C51, batch 512,
        graphed: 2.61 ms per update in fp32, 2.33 with bf16, 1.79 with bf16 + channels-last.
        global_is_max (with process_group): the IS weights of every draw are normalised by the maximum over the
        GLOBAL batch of all ranks (one all-reduce(MAX) of learner_steps floats per draw) instead of per shard.
        replacement=False: every batch holds B distinct records, with the law of the reference's
        torch.multinomial(priority[:top], B, replacement=False) (replay.py:41-43; ReplayDataset.sample), eagerly and
        in the graphed updates.
        publish_weights=True: ``learn`` publishes the online model once after its L updates (weights.WeightPublisher; with
        graph=True the publish is the last node of the captured graph), and ``weight_handle()`` gives what actor
        processes subscribe with (weights.WeightSubscriber).  Off by default: the captured step is then unchanged.
        inbox_lanes=k (with native_nstep=True): the trainer owns an inbox.TransitionInbox of k lanes (``inbox_kw``: its
        slots, slot_transitions, slot_frames); ``inbox_handle(lane)`` gives what an actor process opens a
        TransitionWriter with, and ``step`` drains the inbox into the shard (eagerly, before the updates) where it
        otherwise calls ``extend``.  Off by default."""
        self.pg = process_group
        self.global_is_max = bool(global_is_max) and process_group is not None
        self.cfg = cfg
        self.sampler_seed = sampler_seed
        self.replacement = bool(replacement)
        self.amp = bool(amp)
        self.obs_dtype = torch.bfloat16 if self.amp else None
        self.normalized = NORM_RECIP if (fused_input or self.amp) else None
        self.replay = ReplayDataset(cfg, native_nstep=native_nstep, **replay_kw)
        self.graph = bool(graph)
        self.learner = make_learner(cfg, process_group=process_group, device=self.replay.device,
                                    max_p=None, capturable=self.graph, amp_dtype=torch.bfloat16 if self.amp else None,
                                    channels_last=self.amp if channels_last is None else bool(channels_last))
        self._graphed = None
        self.publisher = None
        if publish_weights:
            from .weights import WeightPublisher
            self.publisher = WeightPublisher(self.learner.model)
        self.inbox = None
        if inbox_lanes:
            if not native_nstep:
                raise ValueError("an inbox feeds the native ingest: construct the Trainer with native_nstep=True")
            from .inbox import TransitionInbox
            self.inbox = TransitionInbox(self.replay, inbox_lanes, **(inbox_kw or {}))
        self.num_transitions = cfg.actor.sample_steps * cfg.actor.num_envs
        self.frame_count = 0
        # the reference keeps every value ever logged (trainer.py:45-47) but only ever reads the last 20 / 100:
        # bounded deques of device scalars, reduced with ONE read-back per step
        self.Ls, self.FLs = deque(maxlen=20), deque(maxlen=20)
        self.Rs, self.Qs = deque(maxlen=20), deque(maxlen=100)
        self.R_max = None

    def learn(self, learner_steps=None):
        """The inner loop (trainer.py:82-109).  Returns per-update (q_loss, fraction_loss) device
        tensors; nothing is synchronised."""
        cfg = self.cfg
        L = int(learner_steps or cfg.learner.learner_steps)
        B = cfg.learner.batch_size
        if self.graph:
            if self._graphed is None or self._graphed.L != L:
                self._graphed = GraphedUpdates(self.learner, self.replay, B, L, normalized=self.normalized,
                                               sampler_seed=self.sampler_seed, obs_dtype=self.obs_dtype,
                                               replacement=self.replacement, publisher=self.publisher)
            return self._graphed.run()
        out = []
        drawn = self.replay.sample(B, k_batches=L, normalized=self.normalized, seed=self.sampler_seed, obs_dtype=self.obs_dtype,
                                   replacement=self.replacement)
        if self.global_is_max and self.replay.prioritize:
            drawn = drawn._replace(weights=self.replay.global_is_weights(drawn.priorities, B, self.pg))
        for b in split_batches(drawn, B):
            result = self.learner.train(_learner_data(b))
            self.replay.update_priority(result["indices"], result["q_loss"])
            out.append((result["q_loss"], result["fraction_loss"]))
        if self.publisher is not None:
            self.publisher.publish()
        return out

    def weight_handle(self):
        """The handle actor processes subscribe to the learner's weights with (``publish_weights=True`` only)."""
        if self.publisher is None:
            raise RuntimeError("construct the Trainer with publish_weights=True to serve weights to actors")
        return self.publisher.handle()

    def inbox_handle(self, lane):
        """The handle an actor process opens lane ``lane`` of the trainer's inbox with (``inbox_lanes`` only)."""
        if self.inbox is None:
            raise RuntimeError("construct the Trainer with inbox_lanes=k to take transitions from actor processes")
        return self.inbox.handle(lane)

    def step(self, transitions=(), returns=(), qmax=()):
        """trainer.py:74-119 with the same argument list: new transitions from the actor (reference
        tuples), episode returns and mean q-values for logging.  With an inbox, the transitions drained from it are
        ingested here and counted into ``frames``."""
        self.Qs.extend(qmax)
        self.Rs.extend(returns)
        self.replay.extend(transitions)
        if self.inbox is not None:
            self.frame_count += self.inbox.drain()
        else:
            self.frame_count += self.num_transitions
        if len(self.replay) > self.cfg.trainer.training_start_steps:
            for q_loss, fraction_loss in self.learn():
                if q_loss is not None:
                    self.Ls.append(q_loss.mean())
                if fraction_loss is not None:
                    self.FLs.append(fraction_loss.mean())
        if returns:
            self.R_max = max(max(returns), self.R_max if self.R_max is not None else max(returns))
        hmean = lambda xs: float(sum(float(x) for x in xs) / len(xs)) if xs else None
        # one device->host read for both loss means (the reference syncs once per update, agent.py:163-169)
        dev = [torch.stack(tuple(xs)).mean() for xs in (self.Ls, self.FLs) if xs]
        vals = torch.stack(dev).tolist() if dev else []
        loss = vals.pop(0) if self.Ls else None
        frac = vals.pop(0) if self.FLs else None
        return dict(frames=self.frame_count, fraction_loss=frac, loss=loss, return_train=hmean(self.Rs),
                    return_train_max=self.R_max, qmax=hmean(self.Qs))

    # ------------------------------------------------------------------ checkpoint
    def _replay_file(self, directory):
        name = "replay.a0ckpt" if self.pg is None else f"replay.rank{torch.distributed.get_rank(self.pg)}.a0ckpt"
        return os.path.join(directory, name)

    def save(self, directory):
        """Checkpoint the run into ``directory``: the shard (``replay.a0ckpt``, ``replay.rank{r}.a0ckpt`` per rank with a
        process group) and ``learner.pt`` -- online and target models, optimizers, update_steps, frame_count, the
        logging deques, R_max and the torch CPU / CUDA and numpy RNG states."""
        os.makedirs(directory, exist_ok=True)
        self.replay.save(self._replay_file(directory))
        if self.pg is not None and torch.distributed.get_rank(self.pg) != 0:
            return
        ln = self.learner
        state = dict(model=ln.model.state_dict(), model_target=ln.model_target.state_dict(), optimizer=ln.optimizer.state_dict(),
                     update_steps=ln.update_steps, frame_count=self.frame_count,
                     logs={k: [float(x) for x in getattr(self, k)] for k in ("Ls", "FLs", "Rs", "Qs")}, R_max=self.R_max,
                     rng_cpu=torch.get_rng_state(), rng_cuda=torch.cuda.get_rng_state(self.replay.device),
                     rng_numpy=np.random.get_state())
        if getattr(ln, "fqf_optimizer", None) is not None:
            state["fqf_optimizer"] = ln.fqf_optimizer.state_dict()
        torch.save(state, os.path.join(directory, "learner.pt"))

    def load(self, directory, rank=None, world=None):
        """Resume from ``save``: into a Trainer built with the same config.  Captured graphs are dropped (the next
        ``learn`` captures again): Adam's state tensors are replaced, and a graph captured before would keep updating
        the old ones.

        ``directory`` may hold ``replay.a0ckpt`` or ``replay.rank0..G-1.a0ckpt`` of a run on G ranks.  When G equals
        this run's world size (``world``, default: the process group's, else 1) and this rank's file (``rank``, default:
        the process group's, else 0) has the shape of its shard, the shard resumes bit for bit (``ReplayDataset.load``).
        Otherwise the files are resharded: this rank merges the streams ``reshard_assignment`` gives it
        (``ReplayDataset.load_merged``), and every Adam param group's eps is set to ``adam_eps`` of the new world (the
        saved state carries the old world's).  A resharded resume continues the run; it is not bit-identical to any
        run, since frame seqs, record positions and the set of streams of each shard change."""
        from .dist import adam_eps
        pg = self.pg
        if rank is None:
            rank = torch.distributed.get_rank(pg) if pg is not None else 0
        if world is None:
            world = torch.distributed.get_world_size(pg) if pg is not None else 1
        files = _replay_files(directory)
        G = len(files)
        rp = self.replay
        own = rp.checkpoint_info(files[rank]) if rank < G else None
        same = own is not None and G == world and (own["N"], own["NF"], own["F"], own["n_step"], own["age_limit"]) == \
            (rp.size, rp.index.NF, rp.F, rp.index.n, rp.index.age_limit)
        if same:
            rp.load(files[rank])
        else:
            ids = [rp.checkpoint_info(f)["streams"] for f in files]
            parts = reshard_assignment(G, world, ids)[rank]
            rp.load_merged([files[f] for f, _ in parts], [m for _, m in parts])
        state = torch.load(os.path.join(directory, "learner.pt"), map_location=self.replay.device, weights_only=False)
        ln = self.learner
        ln.model.load_state_dict(state["model"])
        ln.model_target.load_state_dict(state["model_target"])
        ln.optimizer.load_state_dict(state["optimizer"])
        if "fqf_optimizer" in state:
            ln.fqf_optimizer.load_state_dict(state["fqf_optimizer"])
        ln.update_steps = state["update_steps"]
        self.frame_count = state["frame_count"]
        dev = self.replay.device
        for k, vals in state["logs"].items():
            d = getattr(self, k)
            d.clear()
            d.extend(torch.tensor(v, device=dev) if k in ("Ls", "FLs") else v for v in vals)
        self.R_max = state["R_max"]
        torch.set_rng_state(state["rng_cpu"].cpu())
        torch.cuda.set_rng_state(state["rng_cuda"].cpu(), dev)
        np.random.set_state(state["rng_numpy"])
        if not same:
            for g in ln.optimizer.param_groups:
                g["eps"] = adam_eps(self.cfg.learner.batch_size, world)
        self._graphed = None


def _replay_files(directory):
    """The shard files of a saved run: [replay.a0ckpt] or [replay.rank0.a0ckpt, ..., replay.rank{G-1}.a0ckpt]."""
    one = os.path.join(directory, "replay.a0ckpt")
    if os.path.exists(one):
        return [one]
    files = []
    while os.path.exists(os.path.join(directory, f"replay.rank{len(files)}.a0ckpt")):
        files.append(os.path.join(directory, f"replay.rank{len(files)}.a0ckpt"))
    if not files:
        raise FileNotFoundError(f"{directory} holds no replay.a0ckpt or replay.rank0.a0ckpt")
    return files


def reshard_assignment(G, G_new, stream_ids_per_file):
    """Which streams of G shard files each of G_new ranks takes: a list over the new ranks of [(file, {old id: new
    id})].  G_new <= G: rank r' takes the whole files r with r % G_new == r', the ids of its j-th file offset by j * S
    (S = 1 + the largest id of its files; ReplayDataset.load_merged's default).  G_new > G: rank r' takes file
    r' % G, and of that file's streams in ascending id order (ordinal t) those with t % c == r' // G, where c new ranks
    share the file; ids are kept.  Every (file, stream) goes to exactly one rank."""
    ids = [sorted(int(x) for x in f) for f in stream_ids_per_file]
    assert len(ids) == G and G >= 1 and G_new >= 1
    out = []
    for r2 in range(G_new):
        if G_new <= G:
            mine = [f for f in range(G) if f % G_new == r2]
            S = 1 + max((max(ids[f]) for f in mine if ids[f]), default=-1)
            out.append([(f, {sid: sid + j * S for sid in ids[f]}) for j, f in enumerate(mine)])
        else:
            f = r2 % G
            c = len(range(f, G_new, G))
            out.append([(f, {sid: sid for t, sid in enumerate(ids[f]) if t % c == r2 // G})])
    return out
