"""The sum-tree kernels against the vectorised oracle (oracle/sumtree.py: SumTree.build / .sample / .update) at every
tree depth a shard can have, 1 to 24 (a0_rb_create takes up to 2^24 records), bit for bit:

  (a) the stratified draw (K2a: a0_pt_sample, a0_pt_sample_rng, uniform shards, device-resident scalars) at every
      depth, so that every split between the shared-memory top (10 levels) and the 1..5-level sub-heaps is run, on
      zero runs aligned with the units the descent walks, magnitudes from 2^-20 to 2^20, exact ties and the uniforms
      0 and 1 - 2^-24;
  (b) the priority write-back (every K2b schedule the tree size reaches) at depths 21, 23 and 24, where the chunk
      schedule ends (592 chunks) and where the one-CTA node map runs its 12 sparse levels;
  (c) the fused ingest (a0_k1_append_mark: marks through the same node map) on a 2^24-record shard.

RawShard (16-byte frames) keeps a 2^24-record shard at about 1 GB; one shard per size is made and reused."""
import numpy as np
import pytest
import torch

from agent0_b200 import _lib
from oracle.sumtree import SumTree, philox_uniform
from tests import parity
from tests.test_gpu_sample_unique import RawShard

pytestmark = pytest.mark.gpu
f32 = np.float32
U_MAX = f32(1.0 - 2.0 ** -24)                     # for b >= 1, fl32(b + u) rounds up to b + 1
ALPHA, EPS = 0.5, 0.01
OPT_BULK_MIN, OPT_FUSED_INGEST, OPT_K2B_SMALL, OPT_K2B_CHUNKS, OPT_K2B_SPARSE = 3, 4, 7, 8, 12


@pytest.fixture(scope="module")
def shards():
    made = {}

    def get(N):
        if N not in made:
            made[N] = RawShard(N)
        return made[N]
    yield get
    made.clear()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def _capacity(D, full):
    P = 1 << D
    return P if full else max(2, P - P // 8)


def _leaves(kind, D, N, rng):
    P = 1 << D
    if kind == "spread":
        v = np.sqrt(np.abs(rng.randn(N)) + 0.01)
        v[rng.rand(N) < 0.03] = 0.0
    elif kind.startswith("holes"):
        # zero runs of a sub-heap's bottom (32 leaves), 1024 leaves and everything under one node of the
        # shared-memory top (2^(D-10) leaves), aligned as the descent walks them; "holes_left" also empties the left half
        v = np.sqrt(np.abs(rng.randn(N)) + 0.01)
        for unit in sorted({32, 1024, 1 << max(D - 10, 0)}):
            starts = np.arange(0, N, unit)
            for lo in starts[rng.rand(starts.size) < 0.3]:
                v[lo:lo + unit] = 0.0
        if kind == "holes_left":
            v[:P // 2] = 0.0
        v[N - 1] = 1.0
    elif kind == "range":
        v = np.exp2(rng.uniform(-20, 20, N))
    elif kind == "ties":
        v = np.ones(N)
    elif kind == "first":
        v = np.zeros(N); v[0] = 0.75
    else:                                          # "last"
        v = np.zeros(N); v[N - 1] = 0.75
    return v.astype(f32)


def _load(sh, v):
    """Leaves into the shard (a0_pt_set) and the oracle; the device tree must be the oracle's, node for node."""
    sh.set(torch.arange(v.size, device="cuda"), torch.from_numpy(v).cuda())
    ref = SumTree(sh.N)
    ref.build(v)
    got = sh.tree.cpu().numpy()
    bad = np.flatnonzero(got.view(np.int32) != ref.nodes.view(np.int32))
    assert bad.size == 0, f"{bad.size} tree nodes differ after a0_pt_set, first {bad[:8].tolist()}"
    return ref


def _is_weights(prio, root, top, beta, sum_offset, B):
    """trainer.py:91-94 in float64 from the fp32 priorities and root."""
    w = (top * (prio.astype(np.float64) / (float(root) + sum_offset))) ** -beta
    w = w.reshape(-1, B)
    return (w / (w.max(axis=1, keepdims=True) + 1e-8)).reshape(-1)


class _Out:
    def __init__(self, T):
        self.idx = torch.empty(T, dtype=torch.int64, device="cuda")
        self.prio, self.w, self.u = (torch.empty(T, device="cuda") for _ in range(3))


def _check(ref, o, u, B, top, beta, sum_offset=0.0, uniform=0):
    torch.cuda.synchronize()
    ri, rp = ref.sample(u, B)
    idx, prio, w = o.idx.cpu().numpy(), o.prio.cpu().numpy(), o.w.cpu().numpy()
    assert np.array_equal(idx, ri)
    assert np.array_equal(prio.view(np.int32), rp.view(np.int32))
    assert np.array_equal(prio.view(np.int32), ref.nodes[ref.P + idx].view(np.int32))       # every priority is its leaf
    if ref.root > 0:
        assert (prio > 0).all()
    if uniform:
        assert (w == 1.0).all()
    else:
        parity.close("k2a.weights_all_depths", w, _is_weights(rp, ref.root, top, beta, sum_offset, B))


SHAPES = [(1, 1), (7, 3), (32, 20), (512, 20)]          # single draw; per-warp epilogue; the benchmark's; per-CTA epilogue


@pytest.mark.parametrize("D,full", [(D, False) for D in range(1, 25)] + [(D, True) for D in (10, 15, 20, 24)])
def test_stratified_draw_bit_exact_at_every_depth(shards, D, full):
    N = _capacity(D, full)
    sh = shards(N)
    assert sh.P == 1 << D
    lib, st = sh.lib, _lib.stream_ptr()
    rng = np.random.RandomState(D)
    for kind in ("spread", "holes", "holes_left", "range", "ties", "first", "last"):
        v = _leaves(kind, D, N, rng)
        ref = _load(sh, v)
        top = float(np.count_nonzero(v))
        for B, L in SHAPES:
            T = B * L
            o = _Out(T)
            u_rand = rng.rand(T).astype(f32)
            for u in (u_rand, np.zeros(T, f32), np.full(T, U_MAX)):   # the caller's uniforms
                ud = torch.from_numpy(u).cuda()
                _lib.check(lib.a0_pt_sample(sh.h, ud.data_ptr(), T, B, top, 0.4, 0.0, 0, o.idx.data_ptr(), o.prio.data_ptr(),
                                            o.w.data_ptr(), st), "a0_pt_sample")
                _check(ref, o, u, B, top, 0.4)
            ud = torch.from_numpy(u_rand).cuda()
            _lib.check(lib.a0_pt_sample(sh.h, ud.data_ptr(), T, B, top, 0.4, 0.0, 1, o.idx.data_ptr(), o.prio.data_ptr(),
                                        o.w.data_ptr(), st), "a0_pt_sample")      # uniform shard: weights exactly 1
            _check(ref, o, u_rand, B, top, 0.4, uniform=1)
            # the sampler's own generator: an explicit call number, then twice from the device counter
            seed = 0x5EED_0000 + D
            _lib.check(lib.a0_pt_rng_seek(sh.h, 40 + D, st), "a0_pt_rng_seek")
            for call, want_call in ((7 + D, 7 + D), (-1, 40 + D), (-1, 41 + D)):
                _lib.check(lib.a0_pt_sample_rng(sh.h, seed, call, T, B, top, 0.4, 0.0, 0, o.idx.data_ptr(), o.prio.data_ptr(),
                                                o.w.data_ptr(), o.u.data_ptr(), st), "a0_pt_sample_rng")
                torch.cuda.synchronize()
                want_u = philox_uniform(seed, want_call, T)
                assert np.array_equal(o.u.cpu().numpy(), want_u)
                _check(ref, o, want_u, B, top, 0.4)
            # top / beta / sum_offset resident on the device (top < 0)
            _lib.check(lib.a0_rb_set_dynamic(sh.h, top, 0.7, 12.5, st), "a0_rb_set_dynamic")
            _lib.check(lib.a0_pt_sample(sh.h, ud.data_ptr(), T, B, -1.0, 0.0, 0.0, 0, o.idx.data_ptr(), o.prio.data_ptr(),
                                        o.w.data_ptr(), st), "a0_pt_sample")
            _check(ref, o, u_rand, B, top, 0.7, sum_offset=12.5)


# (chunks, small, bulk_min, sparse) of A0_OPT_K2B_CHUNKS / _SMALL / _BULK_MIN / _SPARSE, as test_gpu_edges forces them
SCHEDULES = {"chunks": (1, 0, 2048, 32), "chunks_full": (1, 0, 2048, 0), "small": (0, 1, 1 << 30, 32),
             "paths": (0, 0, 1 << 30, 32), "bulk": (0, 0, 1, 32)}
DEFAULTS = ((OPT_K2B_CHUNKS, 1), (OPT_K2B_SMALL, 0), (OPT_BULK_MIN, 2048), (OPT_K2B_SPARSE, 32))


def _update_inputs(case, count, P, N, rng):
    if case == "spread_1024":                      # the node map at its design limit: 1024 leaves, 13 keys each
        idx = rng.choice(N, count, replace=False)
    elif case == "subtree_1024":                   # 1024 leaves under one 4096-leaf subtree
        idx = (rng.randint(N // 4096) * 4096) + rng.choice(4096, count, replace=False)
    else:
        idx = rng.randint(-2, P + 2, count)        # out of range on both sides and in [N, P)
        if count > 8:
            idx[-4:] = idx[0]                      # duplicates: the highest k wins ...
            idx[5:7] = (rng.randint(N) & ~1) + np.array([0, 1])     # siblings
            pairs = rng.randint(N // 2, size=count // 8) * 2
            idx[8:8 + 2 * pairs.size:2], idx[9:9 + 2 * pairs.size:2] = pairs, pairs + 1
    loss = (rng.rand(count) * 3).astype(f32)
    if count > 8:
        loss[-1] = np.nan                          # ... and its NaN leaves the old leaf
        idx[2], loss[2], loss[4] = rng.randint(N), np.inf, -0.5
        idx[3], loss[3] = rng.randint(N), 50.0     # the largest finite loss, in the same warp as the infinite one
    return idx.astype(np.int64), loss


@pytest.mark.parametrize("D", [21, 23, 24])
def test_write_back_node_for_node_at_the_deepest_trees(shards, D):
    """Every K2b schedule the tree reaches (the chunk schedule only up to 2^21 leaves), counts around every schedule
    limit, against SumTree.update: the whole tree and max_p, bit for bit."""
    P = 1 << D
    N = _capacity(D, False)
    sh = shards(N)
    lib, st = sh.lib, _lib.stream_ptr()
    max_p = _lib.device_view(lib.a0_rb_ptr(sh.h, _lib.PTR_MAX_P), (1,), "<f4", "cuda", sh.owner)
    rng = np.random.RandomState(D)
    v = np.sqrt(np.abs(rng.randn(N)) + 0.01).astype(f32)
    v[rng.rand(N) < 0.1] = 0.0                                         # evicted since they were sampled
    base_ref = _load(sh, v)
    base = sh.tree.clone()
    cases = [("random", c) for c in (1, 640, 1024, 1025, 16384, 16385)]
    if D == 24:
        cases += [("spread_1024", 1024), ("subtree_1024", 1024)]
    try:
        for name, (chunks, small, bulk_min, sparse) in SCHEDULES.items():
            if chunks and (P >> 12) > 592:
                continue                                               # K2C_MAX_CHUNKS: the other schedules run
            for opt, val in ((OPT_K2B_CHUNKS, chunks), (OPT_K2B_SMALL, small), (OPT_BULK_MIN, bulk_min), (OPT_K2B_SPARSE, sparse)):
                assert lib.a0_set_option(opt, val) == 0
            for case, count in cases:
                idx, loss = _update_inputs(case, count, P, N, rng)
                sh.tree.copy_(base)
                max_p.fill_(0.75)
                ref = SumTree(N)
                ref.nodes = base_ref.nodes.copy()
                want_max = ref.update(idx, loss, EPS, ALPHA, f32(0.75))
                idx_d, loss_d = torch.from_numpy(idx).cuda(), torch.from_numpy(loss).cuda()
                _lib.check(lib.a0_pt_update(sh.h, idx_d.data_ptr(), loss_d.data_ptr(), count, ALPHA, EPS, st), "a0_pt_update")
                torch.cuda.synchronize()
                got = sh.tree.cpu().numpy()
                bad = np.flatnonzero(got.view(np.int32) != ref.nodes.view(np.int32))
                assert bad.size == 0, f"{name} {case} {count}: {bad.size} nodes differ, first {bad[:8].tolist()}"
                assert max_p.cpu().numpy().view(np.int32)[0] == np.array([want_max], f32).view(np.int32)[0], \
                    f"{name} {case} {count}: max_p {float(max_p)} != {float(want_max)}"
    finally:
        for opt, val in DEFAULTS:
            lib.a0_set_option(opt, val)


def test_fused_ingest_marks_at_depth_24():
    """append_steps on a 2^24-record shard: the step-sized ingest marks and unmarks leaves through a0_k1_append_mark's
    node map with 12 sparse levels.  The whole shard state equals the separate launches' (A0_OPT_FUSED_INGEST = 0), the
    tree is the oracle's over the device's leaves, and every leaf marked after the last loss update holds sqrt(max_p)."""
    from tests.test_gpu_edges import _replay, _shard_state, _stream
    lib = _lib.load()
    E, T, n, hw = 8, 60, 3, (16, 16)
    obs, n_new, act, rew, done = _stream(E, T, hw, seed=24, p_new4=0.1, p_static=0.1)
    states = []
    try:
        for fused in (1, 0):
            assert lib.a0_set_option(OPT_FUSED_INGEST, fused) == 0
            rp = _replay(1 << 24, n, E, obs_hw=hw, frame_capacity=400, age_limit=32)
            assert rp.P == 1 << 24
            rp.frames.zero_()
            far = torch.arange(4096, rp.size, 4099, device="cuda")            # live leaves across the tree, so that
            rp.set_priorities(far, torch.full((far.numel(),), 0.5, device="cuda"))   # every sparse level meets a live sibling
            rp.reset_streams(np.arange(E), obs[0])
            for k in range(T):
                new = np.concatenate([obs[k + 1][e, 4 - n_new[k][e]:] for e in range(E)]) if n_new[k].sum() else \
                    np.zeros((0,) + hw, dtype=np.uint8)
                if k % 9 == 0 and k <= 36:                            # losses move max_p between appends
                    live = torch.nonzero(rp.priority.leaves() > 0).view(-1)[:5]
                    rp.update_priority(live, torch.full((len(live),), 1.5 + k, device="cuda"))
                if k == 37:
                    before = (rp.priority.leaves() > 0).cpu().numpy()
                rp.append_steps(np.arange(E), n_new[k], new, act[k], rew[k], done[k])
            assert rp.index.tail_q > 0                                 # records were evicted: unmarks happened
            states.append(_shard_state(rp))
            leaves = states[-1][3][rp.P:rp.P + rp.size]
            ref = SumTree(rp.size)
            ref.build(leaves)
            assert np.array_equal(states[-1][3].view(np.int32), ref.nodes.view(np.int32))
            marked = (leaves > 0) & ~before
            assert marked.sum() >= E
            assert (leaves[marked] == np.sqrt(np.float32(rp.max_p))).all()
            del rp
            torch.cuda.empty_cache()
    finally:
        lib.a0_set_option(OPT_FUSED_INGEST, 1)
    for a, b in zip(*states):
        assert np.array_equal(a, b)
