"""Parity at BASELINE.json's full sizes (2 M-transition shard, 20 x 512 draws) through
size-independent properties -- the oracle's scalar Python loops cannot run there, so besides the vectorised
sum-tree oracle the checker is an independent torch formulation over the raw device state (frames/slots/info/tree
views):

  * gather == frames[slots] rebuilt with torch indexing along the record links (bit-exact),
    n-step returns in float64 with the reference's operation order (bit-exact);
  * every sum-tree node == fl32(left + right); root == what a pairwise fp32 reduction gives;
  * every sampled index is sampleable, its priority is its leaf, the stratified target of draw b
    falls inside the index's prefix interval (float64 check with fp32 slack), and the draw is the vectorised
    oracle's descent of the host copy of the tree, bit for bit;
  * IS weights follow trainer.py:91-94 and max to 1;
  * update_priority is idempotent and order independent; checksum of gathered frames equals the
    checksum of the source frames."""
import numpy as np
import pytest
import torch

from agent0_b200 import _lib
from agent0_b200.config import make_config
from agent0_b200.synth import fill_shard_synthetic
from oracle.sumtree import SumTree, philox_uniform

pytestmark = pytest.mark.gpu
N, E, n, B, K = 2_000_000, 16, 3, 512, 20
FB = 84 * 84


@pytest.fixture(scope="module")
def shard():
    from agent0_b200.replay import ReplayDataset
    cfg = make_config("qr", per=True, n_step=n, batch_size=B, replay_size=N, num_envs=E)
    rp = ReplayDataset(cfg, native_nstep=True)
    fill_shard_synthetic(rp, N + 3 * 65536, E, seed=11)          # wraps the record ring once
    dev = rp.device
    lib = rp.lib
    slots = _lib.device_view(lib.a0_rb_ptr(rp.h, _lib.PTR_REC_SLOTS), (N, 8), "<i4", dev)
    info = _lib.device_view(lib.a0_rb_ptr(rp.h, _lib.PTR_REC_INFO), (N, 4), "<i4", dev)   # {f64 reward, i32 a|d<<31, i32 link}
    g = torch.Generator(device=dev).manual_seed(5)
    pr = (torch.randn(N, device=dev, generator=g).abs() + 0.01).sqrt()
    live = rp.priority.leaves() > 0
    ids = torch.nonzero(live).squeeze(1)
    for lo in range(0, ids.numel(), 1 << 20):
        rp.set_priorities(ids[lo:lo + (1 << 20)], pr[ids[lo:lo + (1 << 20)]])
    torch.cuda.synchronize()
    yield rp, slots, info
    del rp
    torch.cuda.empty_cache()


def test_shard_is_full_and_wrapped(shard):
    rp, slots, info = shard
    assert rp.index.tail_q > 0 and N - 70000 < rp.top <= N
    assert int((rp.priority.leaves() > 0).sum()) == rp.top == int(rp.index.sampleable.sum())


def test_tree_invariants_at_2m_leaves(shard):
    rp, _, _ = shard
    t = rp.tree
    P = rp.P
    assert torch.equal(t[1:P], t[2:2 * P:2] + t[3:2 * P:2])             # every node == fl32(left + right)
    level = t[P:2 * P].clone()
    while level.numel() > 1:
        level = level[0::2] + level[1::2]
    assert level.item() == t[1].item()
    assert t[P + N:2 * P].sum().item() == 0.0                             # padding leaves stay empty


def test_sample_gather_properties_20x512(shard):
    rp, slots, info = shard
    dev = rp.device
    u = torch.rand(B * K, device=dev, generator=torch.Generator(device=dev).manual_seed(9))
    b = rp.sample(B, k_batches=K, u=u)
    idx = b.indices
    leaves = rp.priority.leaves()
    assert bool((leaves[idx] > 0).all()) and torch.equal(b.priorities, leaves[idx])
    # stratified draw: target of draw j of a batch lies inside the prefix interval of its index
    root = rp.tree[1].double()
    cum = torch.cumsum(leaves.double(), 0)
    tgt = ((torch.arange(B * K, device=dev) % B).double() + u.double()) / B * root
    lo_, hi_ = cum[idx] - leaves[idx].double(), cum[idx]
    slack = 2e-6 * root
    assert bool(((tgt >= lo_ - slack) & (tgt <= hi_ + slack)).all())
    ref = SumTree(N)
    ref.build(leaves.cpu().numpy())
    assert np.array_equal(rp.tree.cpu().numpy().view(np.int32), ref.nodes.view(np.int32))
    ref_idx, ref_prio = ref.sample(u.cpu().numpy(), B)
    assert np.array_equal(idx.cpu().numpy(), ref_idx) and np.array_equal(b.priorities.cpu().numpy(), ref_prio)
    # IS weights (trainer.py:91-94) per batch
    w = (rp.top * (b.priorities / rp.tree[1])).pow(-rp.beta).view(K, B)
    w = (w / (w.max(dim=1, keepdim=True)[0] + 1e-8)).view(-1)
    torch.testing.assert_close(b.weights, w, rtol=1e-5, atol=1e-7)
    assert float(b.weights.view(K, B).max(dim=1)[0].min()) > 0.999999
    # gather: rebuild with torch indexing along the links
    p0 = idx
    p1 = info[p0, 3].long()
    p2 = info[p1, 3].long()
    assert bool(((p1 >= 0) & (p2 >= 0)).all())
    sl = torch.cat((slots[p0, :4], slots[p2, 4:]), dim=1).long()
    want = rp.frames[sl.reshape(-1)].view(B * K, 8 * FB)
    assert torch.equal(b.frames, want)
    assert int(b.frames.sum(dtype=torch.int64)) == int(want.sum(dtype=torch.int64))
    rew = lambda p: info[p, :2].contiguous().view(torch.float64).squeeze(1)
    dn = lambda p: (info[p, 2] < 0)
    act = info[p0, 2] & 0x7fffffff
    r = torch.zeros(B * K, dtype=torch.float64, device=dev)
    for p in (p2, p1, p0):                                                # newest -> oldest (agent.py:65-69)
        r = r * 0.99 * (1 - dn(p).double()) + rew(p)
    assert torch.equal(b.rewards.view(torch.int64), r.view(torch.int64))
    assert torch.equal(b.rewards_f32, r.float())
    assert torch.equal(b.terminals, dn(p0) | dn(p1) | dn(p2))
    assert torch.equal(b.actions, act.long())
    assert torch.equal(b.boot_indices, info[p2, 3].long())
    # every distinct frame of a transition shows up wherever it should: stacks overlap by S - n... frames
    same = (sl[:, 3:4] == sl[:, 4:]).any(dim=1)
    assert float(same.float().mean()) > 0.9                               # ordinary steps share frames


def test_update_priority_idempotent_and_order_independent(shard):
    rp, _, _ = shard
    dev = rp.device
    g = torch.Generator(device=dev).manual_seed(3)
    live = torch.nonzero(rp.priority.leaves() > 0).squeeze(1)
    ids = live[torch.randperm(live.numel(), device=dev, generator=g)[:B * K]]
    loss = torch.rand(B * K, device=dev, generator=g) * 4
    rp.update_priority(ids, loss)
    t1 = rp.tree.clone()
    rp.update_priority(ids, loss)                                         # idempotent
    assert torch.equal(rp.tree, t1)
    perm = torch.randperm(B * K, device=dev, generator=g)
    rp.update_priority(ids[perm], loss[perm])                             # order independent (distinct ids)
    assert torch.equal(rp.tree, t1)
    for k in range(K):                                                    # per-batch updates == one big update
        rp.update_priority(ids[k * B:(k + 1) * B], loss[k * B:(k + 1) * B])
    assert torch.equal(rp.tree, t1)
    torch.testing.assert_close(rp.priority.leaves()[ids], (loss + 0.01).sqrt(), rtol=1e-6, atol=0)
    assert rp.max_p >= float(loss.max())
    P = rp.P
    assert torch.equal(rp.tree[1:P], rp.tree[2:2 * P:2] + rp.tree[3:2 * P:2])


def test_sampling_law_at_scale(shard):
    """Draw frequencies over coarse buckets follow the priority mass (the reference's intended
    multinomial law, replay.py:41-43)."""
    rp, _, _ = shard
    dev = rp.device
    leaves = rp.priority.leaves()
    buckets = 64
    edges = torch.linspace(0, N, buckets + 1, device=dev).long()
    mass = torch.stack([leaves[edges[i]:edges[i + 1]].double().sum() for i in range(buckets)])
    mass = mass / mass.sum()
    counts = torch.zeros(buckets, device=dev, dtype=torch.float64)
    draws = 0
    for it in range(20):
        b = rp.sample(B, k_batches=K)
        counts += torch.bincount(torch.bucketize(b.indices, edges[1:-1], right=True), minlength=buckets).double()
        draws += B * K
    freq = counts / draws
    assert float((freq - mass).abs().max()) < 4 * float((mass.max() / draws).sqrt())


def test_duplicates_per_batch_against_the_reference_draw_without_replacement(shard):
    """The reference's sampler interface draws WITHOUT replacement (torch.multinomial(priority[:top], B, False),
    replay.py:41-43: no index twice in a batch, at the price of a law that is no longer P(i) ~ p_i once a heavy
    record has been taken); the stratified tree descent draws WITH replacement and keeps the law.  The figure
    that separates the two is the duplicate rate inside a batch of 512, measured here on three priority
    vectors and recorded by tests/parity.py:
      spread   |N(0,1)|-shaped priorities (the shard as built): no stratum is narrower than a leaf
      peaked   1 % of the records at 100x the rest
      extreme  100 records hold 90 % of the mass (each spans ~4.6 strata: those draws MUST repeat)
    and checked against what the stratification implies: a record of mass m is drawn at most
    ceil(m * B / total) + 1 times per batch."""
    from tests import parity
    rp, _, _ = shard
    dev = rp.device
    leaves = rp.priority.leaves()
    live = torch.nonzero(leaves > 0).squeeze(1)
    saved = leaves[live].clone()
    g = torch.Generator(device=dev).manual_seed(9)
    out = {}

    def measure(tag):
        total = float(rp.priority_sum())
        dup, worst, bound_ok = 0, 0, True
        for it in range(5):
            b = rp.sample(B, k_batches=K, seed=1234, call=it)
            idx = b.indices.view(K, B)
            for k in range(K):
                u, c = torch.unique(idx[k], return_counts=True)
                dup += B - u.numel()
                worst = max(worst, int(c.max()))
                cap = torch.ceil(leaves[u].double() * B / total) + 1
                bound_ok &= bool((c.double() <= cap).all())
        out[tag] = {"duplicate_fraction_per_batch_of_512": round(dup / (5 * K * B), 5), "max_repeats_of_one_record": worst,
                    "reference_multinomial_without_replacement": 0.0}
        assert bound_ok, tag

    try:
        measure("spread")
        ones = torch.ones(live.numel(), device=dev)
        heavy = torch.randperm(live.numel(), device=dev, generator=g)[:live.numel() // 100]
        v = ones.clone(); v[heavy] = 100.0
        for lo in range(0, live.numel(), 1 << 20):
            rp.set_priorities(live[lo:lo + (1 << 20)], v[lo:lo + (1 << 20)])
        measure("peaked_1pct_at_100x")
        v = ones.clone()
        v[heavy[:100]] = 0.9 / 0.1 * float(live.numel() - 100) / 100.0
        for lo in range(0, live.numel(), 1 << 20):
            rp.set_priorities(live[lo:lo + (1 << 20)], v[lo:lo + (1 << 20)])
        measure("extreme_100_records_hold_90pct")
    finally:
        for lo in range(0, live.numel(), 1 << 20):
            rp.set_priorities(live[lo:lo + (1 << 20)], saved[lo:lo + (1 << 20)])
    assert out["spread"]["duplicate_fraction_per_batch_of_512"] < 0.01
    assert out["peaked_1pct_at_100x"]["duplicate_fraction_per_batch_of_512"] < 0.05
    assert 0.5 < out["extreme_100_records_hold_90pct"]["duplicate_fraction_per_batch_of_512"] < 0.9
    parity.RECORD["k2a.duplicates_in_a_batch (with-replacement stratified draw vs replay.py:41-43)"] = out


def test_waved_graphed_step_at_full_size(shard):
    """The default schedule of hotloop.ReplayTargetLoop at BASELINE size (QR-200, 20 x 512 draws on the 2 M shard): the
    gather in 20 waves with the ordered-fetch window on a side stream, each K4 joined to its wave, captured as one CUDA
    graph.  Against the same draw issued as ONE eager gather launch (same sampler seed and call number): indices, stacks,
    n-step scalars, IS weights, losses and gradients bit-identical; the stacks equal the torch rebuild from the raw
    shard; after the step's write-back every tree node is still fl32(left + right)."""
    from agent0_b200.hotloop import ReplayTargetLoop
    rp, slots, info = shard
    dev = rp.device
    T, A, Nq = B * K, 4, 200
    g = torch.Generator(device=dev).manual_seed(21)
    o = {"online": torch.randn(T, A, Nq, device=dev, generator=g) * 3, "tgt_next": torch.randn(T, A, Nq, device=dev, generator=g) * 3,
         "qsel": torch.randn(T, A, device=dev, generator=g)}
    la = ReplayTargetLoop(rp, "qr", B, K, A, o, n_step=n, rng_seed=33, gather_waves=None)
    lb = ReplayTargetLoop(rp, "qr", B, K, A, o, n_step=n, rng_seed=33)
    assert lb.waves is not None and len(lb.waves) == K and lb.window == 400 and la.waves is None
    rp.push_dynamic()
    la.step(update=False); lb.step(update=False)            # warm-up: allocations, function attributes
    torch.cuda.synchronize()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        lb.step(update=False)
    ref = SumTree(N)
    ref.build(rp.priority.leaves().cpu().numpy())
    for call in (700, 701):
        rp.rng_seek(call)
        la.step(update=False)
        rp.rng_seek(call)
        lb.frames.zero_(); lb.loss.fill_(-1.0)
        gr.replay()
        torch.cuda.synchronize()
        for f in ("idx", "prio", "w", "frames", "act", "r64", "r32", "d8", "d32", "boot", "loss", "grad"):
            assert torch.equal(getattr(la, f), getattr(lb, f)), f
        ref_idx, ref_prio = ref.sample(philox_uniform(33, call, T), B)         # the mailbox sampler at depth 21
        assert np.array_equal(lb.idx.cpu().numpy(), ref_idx) and np.array_equal(lb.prio.cpu().numpy(), ref_prio)
    p0 = lb.idx
    p2 = info[info[p0, 3].long(), 3].long()
    sl = torch.cat((slots[p0, :4], slots[p2, 4:]), dim=1).long()
    assert torch.equal(lb.frames, rp.frames[sl.reshape(-1)].view(T, 8 * FB))
    wmax = lb.w.view(K, B).max(dim=1)[0]
    assert float(wmax.min()) > 0.999999 and float(wmax.max()) <= 1.0 and bool(torch.isfinite(lb.loss).all())
    # the whole step, write-back included, as the captured graph bench.py replays
    lb.capture(warm=1)
    root0 = float(rp.tree[1])
    for _ in range(3):
        lb.run()
    torch.cuda.synchronize()
    t, P = rp.tree, rp.P
    assert torch.equal(t[1:P], t[2:2 * P:2] + t[3:2 * P:2]) and float(t[1]) != root0
    leaves = rp.priority.leaves()
    want = (lb.loss + 0.01).sqrt()                         # (loss + eps)^alpha of the last step, later batches win duplicates
    last = {}
    for j, i in enumerate(lb.idx.tolist()):
        last[i] = j
    ii = torch.tensor(list(last.keys()), device=dev)
    jj = torch.tensor(list(last.values()), device=dev)
    torch.testing.assert_close(leaves[ii], want[jj], rtol=1e-6, atol=0)
