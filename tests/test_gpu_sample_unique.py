"""a0_pt_sample_unique (K2a-unique: prioritized batches without replacement, the law of the reference's
torch.multinomial(priority[:top], B, replacement=False), agent0/deepq/replay.py:41-43) against its definition,
oracle/sample_unique.py: indices, priorities and {rounds, candidates} bit-exact, IS weights within the 1e-5
relative contract; then the properties at full size, CUDA-graph replay, the shortfall report and the public surface
(ReplayDataset.sample, hotloop.ReplayTargetLoop, Trainer) with replacement=False."""
import ctypes as C

import numpy as np
import pytest
import torch

from agent0_b200 import _lib
from oracle.sample_unique import sample_unique

pytestmark = pytest.mark.gpu


class RawShard:
    """A shard handle used only for its sum-tree (16-byte frames, 8 of them): tree depths up to 24 cost no frame ring."""

    def __init__(self, capacity):
        self.lib = _lib.load()
        h = C.c_void_p()
        _lib.check(self.lib.a0_rb_create(C.byref(h), capacity, 8, 16, torch.cuda.current_device()), "a0_rb_create")
        self.h, self.N = h, capacity
        self.owner = _lib.HandleOwner(self.lib, h)
        self.P = int(self.lib.a0_rb_tree_leaves(h))
        self.tree = _lib.device_view(self.lib.a0_rb_ptr(h, _lib.PTR_TREE), (2 * self.P,), "<f4", "cuda", self.owner)

    def set(self, ids, values):
        ids = torch.as_tensor(ids, device="cuda", dtype=torch.int64).contiguous()
        values = torch.as_tensor(values, device="cuda", dtype=torch.float32).contiguous()
        for lo in range(0, ids.numel(), 1 << 20):
            _lib.check(self.lib.a0_pt_set(self.h, ids[lo:lo + (1 << 20)].data_ptr(), values[lo:lo + (1 << 20)].data_ptr(),
                                          min(1 << 20, ids.numel() - lo), _lib.stream_ptr()), "a0_pt_set")
        torch.cuda.synchronize()

    def draw(self, seed, call, K, B, top, beta=0.4, sum_offset=0.0, uniform=0, check=True):
        idx = torch.empty(K * B, dtype=torch.int64, device="cuda")
        prio, w = torch.empty(K * B, device="cuda"), torch.empty(K * B, device="cuda")
        st = torch.full((K, 2), -1, dtype=torch.int32, device="cuda")
        rc = self.lib.a0_pt_sample_unique(self.h, seed, call, K * B, B, top, beta, sum_offset, uniform, idx.data_ptr(),
                                          prio.data_ptr(), w.data_ptr(), st.data_ptr(), _lib.stream_ptr())
        if check:
            _lib.check(rc, "a0_pt_sample_unique")
        return idx, prio, w, st, rc

    def seek(self, call):
        _lib.check(self.lib.a0_pt_rng_seek(self.h, call, _lib.stream_ptr()), "a0_pt_rng_seek")


def priorities(kind, n, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    if kind == "spread":
        return (torch.randn(n, device="cuda", generator=g).abs() + 0.01).sqrt()
    v = torch.ones(n, device="cuda")
    perm = torch.randperm(n, device="cuda", generator=g)
    if kind == "peaked":                                     # 1 % of the records at 100x the rest
        v[perm[:max(1, n // 100)]] = 100.0
        return v
    h = min(100, max(1, n // 10))                            # `h` records (100 when n allows) hold 90 % of the mass
    v[perm[:h]] = 0.9 / 0.1 * float(n - h) / h
    return v


def _fill(sh, kind, live_frac=1.0, seed=0):
    n = sh.N
    v = priorities(kind, n, seed)
    if live_frac < 1.0:
        g = torch.Generator(device="cuda").manual_seed(seed + 1)
        v[torch.rand(n, device="cuda", generator=g) >= live_frac] = 0.0
    sh.set(torch.arange(n, device="cuda"), v)
    return int((v > 0).sum())


def _check_oracle(sh, seed, call, K, B, top, beta=0.4, sum_offset=0.0, uniform=0, got=None, name="k2a_unique.weights"):
    from tests import parity
    idx, prio, w, st, _ = got if got is not None else sh.draw(seed, call, K, B, top, beta, sum_offset, uniform)
    torch.cuda.synchronize()
    nodes = sh.tree.cpu().numpy()
    ri, rp_, rw, rs, short = sample_unique(nodes, sh.P, seed, call, K, B, top=top, beta=beta, sum_offset=sum_offset,
                                           uniform=bool(uniform))
    assert not short.any()
    np.testing.assert_array_equal(idx.cpu().numpy(), ri)
    np.testing.assert_array_equal(prio.cpu().numpy(), rp_)
    np.testing.assert_array_equal(st.cpu().numpy(), rs)
    parity.close(name, w, rw)
    return ri, rs


@pytest.mark.parametrize("D,B,K", [(1, 2, 3), (3, 4, 5), (11, 64, 6), (17, 512, 4), (22, 512, 20), (24, 512, 20)])
@pytest.mark.parametrize("kind", ["spread", "peaked", "extreme"])
def test_bit_exact_against_the_oracle(D, B, K, kind):
    sh = RawShard(1 << D)
    live = _fill(sh, kind, live_frac=0.97 if D >= 11 else 1.0, seed=D)
    for call in (0, 7):
        ri, rs = _check_oracle(sh, 1234 + D, call, K, B, float(live), beta=0.5)
        rows = ri.reshape(K, B)
        assert all(len(np.unique(r)) == B for r in rows)
        leaves = sh.tree[sh.P:].cpu().numpy()
        assert (leaves[ri] > 0).all()


def test_uniform_shard_dynamic_scalars_and_device_call_counter():
    sh = RawShard(3000)
    sh.set(torch.arange(2900, device="cuda"), torch.ones(2900, device="cuda"))
    _check_oracle(sh, 5, 3, 8, 128, 2900.0, uniform=1)
    # top < 0: top / beta / sum_offset published on the device (a0_rb_set_dynamic)
    _fill(sh, "peaked", seed=4)
    _lib.check(sh.lib.a0_rb_set_dynamic(sh.h, 2500.0, 0.7, 12.0, _lib.stream_ptr()), "a0_rb_set_dynamic")
    got = sh.draw(9, 2, 4, 100, -1.0)
    _check_oracle(sh, 9, 2, 4, 100, 2500.0, beta=0.7, sum_offset=12.0, got=got)
    # call < 0: the device counter (a0_pt_rng_seek), advanced once per launch
    sh.seek(41)
    for call in (41, 42, 43):
        got = sh.draw(9, -1, 4, 100, 3000.0)
        _check_oracle(sh, 9, call, 4, 100, 3000.0, got=got)
    explicit = sh.draw(9, 44, 4, 100, 3000.0)
    assert torch.equal(sh.draw(9, -1, 4, 100, 3000.0)[0], explicit[0])


def test_captured_graph_replays_draw_fresh_batches():
    sh = RawShard(1 << 12)
    _fill(sh, "extreme", seed=8)
    K, B = 3, 256
    idx = torch.empty(K * B, dtype=torch.int64, device="cuda")
    prio, w = torch.empty(K * B, device="cuda"), torch.empty(K * B, device="cuda")
    st = torch.empty((K, 2), dtype=torch.int32, device="cuda")
    sh.seek(0)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        _lib.check(sh.lib.a0_pt_sample_unique(sh.h, 77, -1, K * B, B, 4096.0, 0.4, 0.0, 0, idx.data_ptr(), prio.data_ptr(),
                                              w.data_ptr(), st.data_ptr(), _lib.stream_ptr()), "a0_pt_sample_unique")
    seen = []
    for call in range(3):
        g.replay()
        _check_oracle(sh, 77, call, K, B, 4096.0, got=(idx, prio, w, st, 0))
        seen.append(idx.clone())
    assert not torch.equal(seen[0], seen[1]) and not torch.equal(seen[1], seen[2])


def test_shortfall_reports_fault_code_2_and_returns_valid_rows():
    sh = RawShard(2048)
    live = _fill(sh, "spread", seed=2)
    B = 64
    saved = sh.tree[sh.P:sh.P + sh.N].clone()
    try:
        keep = torch.arange(0, 2048, 31, device="cuda")[:B - 1]          # B - 1 positive leaves
        z = torch.ones(2048, dtype=torch.bool, device="cuda")
        z[keep] = False
        sh.set(torch.nonzero(z).squeeze(1), torch.zeros(int(z.sum()), device="cuda"))
        idx, prio, w, st, rc = sh.draw(3, 0, 2, B, float(live))
        torch.cuda.synchronize()                                          # the launch ends
        assert rc == 0
        idx_h = idx.view(2, B).cpu()
        for r in idx_h:
            assert sorted(set(r[:B - 1].tolist())) == sorted(keep.tolist())
            assert (r[B - 1:] == r[0]).all()
        assert (prio > 0).all()
        rc = sh.draw(3, 1, 2, B, float(live), check=False)[4]
        assert rc == -3                                                   # A0_EFAULT
        msg = sh.lib.a0_last_error()
        assert b"fault 2" in msg and b"fewer than B records" in msg
        assert sh.draw(3, 1, 1, B - 1, float(live), check=False)[4] == 0  # reported once
    finally:
        sh.set(torch.arange(sh.N, device="cuda"), saved)
        torch.cuda.synchronize()
        sh.lib.a0_rb_check_fault(sh.h)


def test_full_size_no_duplicates_first_draw_law_and_duplicate_record():
    """2 M records, 20 x 512 per call: no index twice in a batch, every index a live record, and the FIRST draw of
    each batch follows p over 64 buckets (the first draw of successive sampling has law p).  The duplicate
    fraction is recorded beside the stratified draw's figures (test_gpu_fullsize)."""
    from tests import parity
    N, B, K = 2_000_000, 512, 20
    sh = RawShard(N)
    out = {}
    for kind in ("spread", "peaked", "extreme"):
        live = _fill(sh, kind, live_frac=0.95, seed=21)
        leaves = sh.tree[sh.P:sh.P + N]
        dup, rounds, cands = 0, [], []
        for call in range(5):
            idx, prio, w, st, _ = sh.draw(1234, call, K, B, float(live))
            rows = idx.view(K, B)
            dup += sum(B - int(torch.unique(rows[k]).numel()) for k in range(K))
            assert bool((leaves[idx] > 0).all()) and torch.equal(prio, leaves[idx])
            rounds.append(st[:, 0].float().mean().item()); cands.append(st[:, 1].float().mean().item())
        tag = {"spread": "spread", "peaked": "peaked_1pct_at_100x", "extreme": "extreme_100_records_hold_90pct"}[kind]
        out[tag] = {"duplicate_fraction_per_batch_of_512": dup / (5 * K * B), "mean_rounds": round(float(np.mean(rounds)), 3),
                     "mean_candidates_per_batch": round(float(np.mean(cands)), 1)}
        assert dup == 0
    parity.RECORD["k2a_unique.duplicates_in_a_batch (draw without replacement, replay.py:41-43)"] = out
    # first draw of every batch over 64 buckets, under the spread priorities
    _fill(sh, "spread", live_frac=0.95, seed=21)
    leaves = sh.tree[sh.P:sh.P + N]
    edges = torch.linspace(0, N, 65, device="cuda").long()
    mass = torch.stack([leaves[edges[i]:edges[i + 1]].double().sum() for i in range(64)])
    mass = mass / mass.sum()
    counts = torch.zeros(64, dtype=torch.float64, device="cuda")
    calls = 100
    for call in range(calls):
        first = sh.draw(99, call, K, B, float(N))[0].view(K, B)[:, 0].contiguous()
        counts += torch.bincount(torch.bucketize(first, edges[1:-1], right=True), minlength=64).double()
    freq = counts / (calls * K)
    assert float((freq - mass).abs().max()) < 4 * float((mass.max() / (calls * K)).sqrt())


# ---------------------------------------------------------------------------------------------- public surface
B_, L_, A_ = 16, 3, 4


def _replay(seed=3):
    from agent0_b200.config import make_config
    from agent0_b200.replay import ReplayDataset
    from agent0_b200.synth import fill_shard_synthetic
    cfg = make_config("c51", per=True, n_step=3, batch_size=B_, replay_size=4096, double_q=True, dueling=True, num_envs=8,
                      action_dim=A_)
    rp = ReplayDataset(cfg, native_nstep=True)
    fill_shard_synthetic(rp, 4096, 8, seed)
    ids = torch.arange(0, 4000, 7, device="cuda")
    rp.update_priority(ids, torch.rand(len(ids), device="cuda", generator=torch.Generator("cuda").manual_seed(seed)) * 40)
    return rp


def test_replay_dataset_sample_without_replacement():
    rp = _replay()
    st = torch.empty((L_, 2), dtype=torch.int32, device="cuda")
    b = rp.sample(B_, k_batches=L_, seed=5, call=2, replacement=False, stats_out=st)
    ri, _, rw, rs, _ = sample_unique(rp.tree.cpu().numpy(), rp.P, 5, 2, L_, B_, top=rp.top, beta=rp.beta)
    np.testing.assert_array_equal(b.indices.cpu().numpy(), ri)
    np.testing.assert_array_equal(st.cpu().numpy(), rs)
    from tests import parity
    parity.close("k2a_unique.weights", b.weights, rw)
    assert torch.equal(b.frames, rp.gather(b.indices).frames)
    # without a seed: one 64-bit seed drawn from the generator and kept; the device counter advances
    torch.manual_seed(0)
    b1 = rp.sample(B_, k_batches=L_, replacement=False)
    b2 = rp.sample(B_, k_batches=L_, replacement=False)
    assert not torch.equal(b1.indices, b2.indices)
    for b in (b1, b2):
        assert all(len(set(r)) == B_ for r in b.indices.view(L_, B_).tolist())
    with pytest.raises(ValueError):
        rp.sample(B_, replacement=False, u=torch.rand(B_, device="cuda"))
    with pytest.raises(ValueError):
        rp.sample(B_, replacement=False, indices=torch.arange(B_, device="cuda"))
    with pytest.raises(ValueError):
        rp.sample(2048, replacement=False)


def test_prebound_loop_without_replacement_equals_the_general_api():
    """ReplayTargetLoop(replacement=False), eager and graph-replayed, against ReplayDataset.sample(replacement=False)
    + losses.c51_loss + update_priority on a twin shard: indices, weights, stacks, losses, gradients, the tree."""
    from agent0_b200 import losses as LS
    from agent0_b200.hotloop import ReplayTargetLoop
    from agent0_b200.replay import split_batches
    T = B_ * L_
    g = torch.Generator(device="cuda").manual_seed(7)
    rn = lambda *s: torch.randn(*s, device="cuda", generator=g) * 3.0
    o = {"qsel": rn(T, A_), "online": rn(T, A_, 51), "tgt_next": rn(T, A_, 51), "atoms": torch.linspace(-10, 10, 51, device="cuda")}
    rp_a, rp_b, rp_c = _replay(), _replay(), _replay()
    b = rp_a.sample(B_, k_batches=L_, seed=19, call=0, replacement=False)
    gam = float(np.float32(0.99 ** 3))
    outs, grads = [], []
    for k, bk in enumerate(split_batches(b, B_)):
        s = slice(k * B_, (k + 1) * B_)
        r = LS.c51_loss(o["online"][s], o["tgt_next"][s], o["atoms"], bk.actions, bk.rewards_f32, bk.terminals_f32, bk.weights,
                        gam, -10.0, 10.0, qsel=o["qsel"][s], max_p=rp_a.max_p_tensor)
        outs.append(r.loss); grads.append(r.grad)
    loss_ref, grad_ref = torch.cat(outs), torch.cat(grads)
    rp_a.update_priority(b.indices, loss_ref)
    with pytest.raises(ValueError):
        ReplayTargetLoop(rp_b, "c51", B_, L_, A_, o, n_step=3, replacement=False, overlap_sample_gather=True)
    for rp, graph in ((rp_b, False), (rp_c, True)):
        loop = ReplayTargetLoop(rp, "c51", B_, L_, A_, o, n_step=3, rng_seed=19, replacement=False)
        assert loop.waves is None and not loop.overlap_sg
        rp.push_dynamic()
        rp.rng_seek(0)
        if graph:
            loop.idx.zero_()
            loop.gather()
            torch.cuda.synchronize()
            cg = torch.cuda.CUDAGraph()
            with torch.cuda.graph(cg):
                loop.step()
            cg.replay()
        else:
            loop.step()
        torch.cuda.synchronize()
        assert torch.equal(loop.idx, b.indices) and torch.equal(loop.w, b.weights)
        assert torch.equal(loop.frames, b.frames) and torch.equal(loop.r64, b.rewards)
        assert torch.equal(loop.loss, loss_ref) and torch.equal(loop.grad, grad_ref)
        assert torch.equal(rp.tree, rp_a.tree) and float(rp.max_p_tensor) == float(rp_a.max_p_tensor)


def test_trainer_graphed_c51_update_without_replacement(golden):
    from agent0_b200.config import make_config
    from agent0_b200.trainer import Trainer
    g = golden("replay_n3")
    M = len(g["entry_action"])
    tup = [(g["entry_frames"][i].tobytes(), g["entry_action"][i], g["entry_reward"][i], g["entry_done"][i]) for i in range(M)]
    cfg = make_config("c51", per=True, n_step=3, batch_size=8, double_q=True, dueling=True, replay_size=256, num_envs=3)
    cfg.trainer.training_start_steps = 10
    cfg.learner.learner_steps = 4
    cfg.learner.target_update_freq = 8
    torch.manual_seed(11)
    tr = Trainer(cfg, graph=True, sampler_seed=31, replacement=False)
    tr.replay.extend(tup)
    seen = []
    for step in range(3):
        out = tr.learn()
        torch.cuda.synchronize()
        assert all(bool(torch.isfinite(q).all()) for q, _ in out)
        rows = tr._graphed.static.indices.view(4, 8).cpu()
        assert all(len(set(r.tolist())) == 8 for r in rows)
        seen.append(rows.clone())
    assert tr.learner.update_steps == 12
    assert not torch.equal(seen[1], seen[2])                  # the replayed draw advances the device call counter
