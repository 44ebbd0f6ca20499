"""K1/K2/K3 parity on the GPU through the C ABI (via agent0_b200.replay.ReplayDataset).

Bit-exact: gathered uint8 stacks, actions, n-step returns (float64 bits), done flags, bootstrap
indices, sampled indices and the whole sum-tree.  <=1e-5 relative: IS weights, priorities."""
import numpy as np
import pytest
import torch

from agent0_b200.config import make_config
from agent0_b200.synth import record_stream
from oracle import reference_replay as OR
from oracle.sumtree import SumTree, new_priority

pytestmark = pytest.mark.gpu
FG = 84 * 84


def _np(t):
    return t.detach().cpu().numpy()


def _replay(size, n=1, per=True, native=False, E=3, **kw):
    from agent0_b200.replay import ReplayDataset
    cfg = make_config("c51", per=per, n_step=n, batch_size=8, replay_size=size, num_envs=E)
    cfg.trainer.total_steps = 1000
    return ReplayDataset(cfg, native_nstep=native, **kw)


def _tuples(g, lo, hi):
    return [(g["entry_frames"][i].tobytes(), g["entry_action"][i], g["entry_reward"][i], g["entry_done"][i])
            for i in range(lo, hi)]


@pytest.mark.parametrize("n", [1, 3])
@pytest.mark.parametrize("variant", [0, 1, 2, 3])
def test_extend_then_gather_equals_reference_getitem(golden, n, variant):
    """ReplayDataset.extend(reference tuples) -> gather(i) == reference replay[i] (replay.py:32-37)."""
    g = golden(f"replay_n{n}")
    M = len(g["entry_action"])
    rp = _replay(256, n=n, gather_variant=variant)
    for lo in range(0, M, 45):
        rp.extend(_tuples(g, lo, min(M, lo + 45)))
    assert len(rp) == rp.top == M
    b = rp.gather(torch.arange(M, device="cuda"))
    assert np.array_equal(_np(b.frames), g["entry_frames"])
    assert np.array_equal(_np(b.actions), g["entry_action"])
    assert np.array_equal(_np(b.rewards).view(np.int64), g["entry_reward"].view(np.int64))
    assert np.array_equal(_np(b.terminals), g["entry_done"])
    assert np.array_equal(_np(b.rewards_f32), g["entry_reward"].astype(np.float32))
    assert np.array_equal(_np(b.terminals_f32), g["entry_done"].astype(np.float32))
    assert b.frames.dtype == torch.uint8 and b.actions.dtype == torch.int64
    assert b.rewards.dtype == torch.float64 and b.terminals.dtype == torch.bool


def test_extend_accepts_lz4_blocks_ndarrays_and_bytes(golden):
    """The reference actor ships lz4.block.compress(concat(st, st_next)) (agent.py:78-81): python-lz4
    block framing (4-byte size prefix) decoded through the system liblz4 straight into the ingest
    buffer; raw bytes and ndarrays are accepted too.  Several extend() calls, mixed formats."""
    from oracle import cpu_path as CP
    g = golden("replay_n3")
    z = CP.lz4()
    M = len(g["entry_action"])
    rp = _replay(256, n=1, E=int(g["num_envs"]))
    tup = []
    for i in range(M):
        raw = g["entry_frames"][i].tobytes()
        blob = (z.compress(raw), raw, g["entry_frames"][i])[i % 3]
        tup.append((blob, g["entry_action"][i], g["entry_reward"][i], g["entry_done"][i]))
    assert len(tup[0][0]) < 56448 // 4                          # really compressed
    for lo in range(0, M, 37):
        rp.extend(tup[lo:lo + 37], streams=np.arange(lo, min(M, lo + 37)) % int(g["num_envs"]))
    assert rp.top == M and rp.index.head_fs < 3 * M             # de-duplicated: ~1-2 stored frames per entry, not 8
    b = rp.gather(torch.arange(M, device="cuda"))
    assert np.array_equal(_np(b.frames), g["entry_frames"])
    assert np.array_equal(_np(b.actions), g["entry_action"]) and np.array_equal(_np(b.terminals), g["entry_done"])
    assert np.array_equal(_np(b.rewards).view(np.int64), g["entry_reward"].view(np.int64))


@pytest.mark.parametrize("n", [1, 3])
def test_native_nstep_gather_equals_reference_actor_entries(golden, n):
    """Raw 1-step transitions in; K3 folds n steps: must equal Actor.sample's entries
    (agent.py:64-81) under the Appendix-C index mapping."""
    g = golden(f"replay_n{n}")
    E, T = int(g["num_envs"]), int(g["steps"])
    obs = g["stream_obs"]
    done = OR.done_rule(g["stream_terminal"], g["stream_life_loss"], g["stream_truncated"])
    for variant in (0, 1, 2, 3):
        rp = _replay(256, n=n, native=True, E=E, gather_variant=variant)
        for k in range(T):
            rp.append_vector_step(obs[k], g["stream_action"][k], g["stream_reward"][k], done[k], obs[k + 1])
        assert rp.top == (T - n + 1) * E
        ks, es = np.meshgrid(np.arange(n - 1, T), np.arange(E), indexing="ij")
        ref_i = (ks * E + es).reshape(-1)
        pos = ((ks - n + 1) * E + es).reshape(-1)
        b = rp.gather(torch.as_tensor(pos, device="cuda"))
        assert np.array_equal(_np(b.frames), g["entry_frames"][ref_i])
        assert np.array_equal(_np(b.actions), g["entry_action"][ref_i])
        assert np.array_equal(_np(b.rewards).view(np.int64), g["entry_reward"][ref_i].view(np.int64))
        assert np.array_equal(_np(b.terminals), g["entry_done"][ref_i])
        boot = np.where(ks + 1 < T, (ks + 1) * E + es, -1).reshape(-1)
        assert np.array_equal(_np(b.boot_indices), boot)


def test_device_resident_native_ingest_and_wraparound():
    """Frames already on the GPU, ring smaller than the stream: every sampleable record must
    gather what the brute-force history says (oracle pack_nstep), TMA and LDG variants alike."""
    E, T, n = 4, 90, 3
    s = record_stream(E, T, seed=77, p_terminal=0.05, p_life_loss=0.05, p_truncated=0.03)
    fr_ref, a_ref, r_ref, d_ref = OR.pack_nstep(s["obs"], s["action"], s["reward"], s["done"], n, 0.99)
    from agent0_b200.ring_index import stack_delta
    rp = _replay(96, n=n, native=True, E=E, frame_capacity=400, age_limit=32)
    rp.reset_streams(np.arange(E), torch.as_tensor(s["obs"][0]).cuda())
    for k in range(T):
        kk = stack_delta(s["obs"][k], s["obs"][k + 1])
        new = np.concatenate([s["obs"][k + 1][e, 4 - kk[e]:] for e in range(E)])
        rp.append_steps(np.arange(E), kk, torch.as_tensor(new).cuda(), s["action"][k], s["reward"][k], s["done"][k])
    ix = rp.index
    assert ix.tail_q > 0
    leaves = _np(rp.priority.leaves())
    live = np.flatnonzero(leaves > 0)
    assert len(live) == rp.top and np.array_equal(live, np.flatnonzero(ix.sampleable))
    q = ix.head_q - 1 - ((ix.head_q - 1 - live) % rp.size)
    k0, e = np.divmod(q, E)
    ref_i = (k0 + n - 1) * E + e
    for variant in (0, 1, 2, 3):
        rp.gather_variant = variant
        b = rp.gather(torch.as_tensor(live, device="cuda"))
        assert np.array_equal(_np(b.frames), fr_ref[ref_i])
        assert np.array_equal(_np(b.rewards).view(np.int64), r_ref[ref_i].view(np.int64))
        assert np.array_equal(_np(b.terminals), d_ref[ref_i]) and np.array_equal(_np(b.actions), a_ref[ref_i])


@pytest.mark.parametrize("mode", ["pageable", "pinned", "pinned_copy_stream", "pageable_copy_stream"])
def test_host_fed_ingest_modes_and_wraparound(mode):
    """New frames arriving from HOST memory (pageable staging, pinned DMA, and either of them on the
    shard's copy stream while the main stream is busy): same ring contents as the brute-force history."""
    E, T, n = 4, 90, 3
    s = record_stream(E, T, seed=78, p_terminal=0.05, p_life_loss=0.05, p_truncated=0.03)
    fr_ref, a_ref, r_ref, d_ref = OR.pack_nstep(s["obs"], s["action"], s["reward"], s["done"], n, 0.99)
    from agent0_b200.ring_index import stack_delta
    rp = _replay(96, n=n, native=True, E=E, frame_capacity=400, age_limit=32)
    rp.reset_streams(np.arange(E), s["obs"][0])
    busy = torch.empty(1 << 24, device="cuda")
    keep = []
    for k in range(T):
        kk = stack_delta(s["obs"][k], s["obs"][k + 1])
        new = torch.as_tensor(np.concatenate([s["obs"][k + 1][e, 4 - kk[e]:] for e in range(E)]))
        pinned = mode.startswith("pinned")
        if pinned:
            new = new.pin_memory()
            keep.append(new)
        busy.normal_()                      # keeps the main stream busy so the side-stream DMA really overlaps
        rp.append_steps(np.arange(E), kk, new, s["action"][k], s["reward"][k], s["done"][k], pinned_stable=pinned,
                        copy_stream=mode.endswith("copy_stream"))
    ix = rp.index
    assert ix.tail_q > 0
    live = np.flatnonzero(_np(rp.priority.leaves()) > 0)
    assert len(live) == rp.top and np.array_equal(live, np.flatnonzero(ix.sampleable))
    q = ix.head_q - 1 - ((ix.head_q - 1 - live) % rp.size)
    k0, e = np.divmod(q, E)
    ref_i = (k0 + n - 1) * E + e
    b = rp.gather(torch.as_tensor(live, device="cuda"))
    assert np.array_equal(_np(b.frames), fr_ref[ref_i])
    assert np.array_equal(_np(b.rewards).view(np.int64), r_ref[ref_i].view(np.int64))
    assert np.array_equal(_np(b.terminals), d_ref[ref_i]) and np.array_equal(_np(b.actions), a_ref[ref_i])


def _norm_ref(u8, mode):
    """agent.py:129-135 / trainer.py:88-90 on the host: mode 0 = torch-CPU true division, 1 = torch-CUDA
    reciprocal multiply, 2 = .float() only; all float32."""
    x = u8.astype(np.float32)
    if mode == 0:
        return x / np.float32(255.0)
    if mode == 1:
        return x * (np.float32(1.0) / np.float32(255.0))
    return x


@pytest.mark.parametrize("n", [1, 3])
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_fused_f32_gather_equals_reference_float_div_split(golden, n, mode):
    """a0_rb_gather_f32 = K3 + BaseLearner.train's reshape/.float()/.div(255)/split (agent.py:129-135):
    bit-exact f32 against the reference actor's entries converted on the host, scalars as K3."""
    g = golden(f"replay_n{n}")
    E, T = int(g["num_envs"]), int(g["steps"])
    obs = g["stream_obs"]
    done = OR.done_rule(g["stream_terminal"], g["stream_life_loss"], g["stream_truncated"])
    rp = _replay(256, n=n, native=True, E=E)
    for k in range(T):
        rp.append_vector_step(obs[k], g["stream_action"][k], g["stream_reward"][k], done[k], obs[k + 1])
    ks, es = np.meshgrid(np.arange(n - 1, T), np.arange(E), indexing="ij")
    ref_i = (ks * E + es).reshape(-1)
    pos = torch.as_tensor(((ks - n + 1) * E + es).reshape(-1), device="cuda")
    b = rp.gather(pos, normalized=mode)
    assert b.frames is None and b.obs.dtype == torch.float32 and b.obs.shape == (len(ref_i), 4, 84, 84)
    ref = _norm_ref(g["entry_frames"][ref_i].reshape(-1, 8, 84, 84), mode)
    assert np.array_equal(_np(b.obs).view(np.int32), ref[:, :4].view(np.int32))
    assert np.array_equal(_np(b.next_obs).view(np.int32), ref[:, 4:].view(np.int32))
    assert np.array_equal(_np(b.actions), g["entry_action"][ref_i])
    assert np.array_equal(_np(b.rewards).view(np.int64), g["entry_reward"][ref_i].view(np.int64))
    assert np.array_equal(_np(b.terminals), g["entry_done"][ref_i])
    # the u8 gather + torch's own cast/divide on this device gives the same bits as mode 1
    if mode == 1:
        u = rp.gather(pos).frames.reshape(-1, 8, 84, 84).float().div(255.0)
        assert torch.equal(u[:, :4], b.obs) and torch.equal(u[:, 4:], b.next_obs)


def test_fused_f32_gather_every_byte_value_and_out_buffers():
    """All 256 byte values through the three normalisations; preallocated out= buffers; error paths."""
    from agent0_b200.replay import NORM_DIV
    E = 2
    rp = _replay(64, n=1, native=True, E=E)
    ramp = (np.arange(4 * 84 * 84, dtype=np.int64) % 256).astype(np.uint8).reshape(4, 84, 84)
    obs0 = np.stack([ramp, ramp[::-1].copy()])
    rp.reset_streams(np.arange(E), obs0)
    new = np.stack([np.full((84, 84), 255, np.uint8), np.zeros((84, 84), np.uint8)])
    rp.append_steps(np.arange(E), np.ones(E, dtype=np.int64), new, np.array([1, 2]), np.array([0.5, -1.0]), np.array([False, True]))
    pos = torch.arange(E, device="cuda")
    u8 = _np(rp.gather(pos).frames).reshape(E, 8, 84, 84)
    for mode in (0, 1, 2):
        b = rp.gather(pos, normalized=mode)
        ref = _norm_ref(u8, mode)
        assert np.array_equal(_np(b.obs), ref[:, :4]) and np.array_equal(_np(b.next_obs), ref[:, 4:])
    out = rp.alloc_batch(E, normalized=NORM_DIV)
    b = rp.sample(E, indices=pos, out=out)
    assert b.obs.data_ptr() == out.obs.data_ptr() and np.array_equal(_np(out.obs), _norm_ref(u8, 0)[:, :4])
    with pytest.raises(RuntimeError, match="norm_mode"):
        rp.gather(pos, normalized=7)


def test_sumtree_sample_update_bit_exact():
    """K2a/K2b against oracle/sumtree.py: same leaves, same uniforms -> identical indices and an
    identical tree, node for node."""
    N = 5000
    rp = _replay(N, per=True)
    rng = np.random.RandomState(0)
    pr = ((np.abs(rng.randn(N)) + 0.01) ** 0.5).astype(np.float32)
    pr[rng.rand(N) < 0.3] = 0.0
    ref = SumTree(N)
    ref.set(np.arange(N), pr)
    rp.set_priorities(torch.arange(N), torch.as_tensor(pr))
    assert np.array_equal(_np(rp.tree)[:2 * ref.P], ref.nodes)
    import types
    rp.index = types.SimpleNamespace(top=int((pr > 0).sum()))      # leaves were set directly, not appended
    for B, K in ((32, 1), (512, 1), (32, 20), (7, 3)):
        u = rng.rand(B * K).astype(np.float32)
        idx = torch.empty(B * K, dtype=torch.int64, device="cuda")
        prio = torch.empty(B * K, device="cuda"); w = torch.empty(B * K, device="cuda")
        from agent0_b200 import _lib
        u_dev = torch.as_tensor(u).cuda()
        _lib.check(rp.lib.a0_pt_sample(rp.h, u_dev.data_ptr(), B * K, B, float(rp.top), 0.6,
                                       0.0, 0, idx.data_ptr(), prio.data_ptr(), w.data_ptr(),
                                       _lib.stream_ptr()), "a0_pt_sample")
        for k in range(K):
            ridx, rprio = ref.sample_stratified(u[k * B:(k + 1) * B])
            assert np.array_equal(_np(idx)[k * B:(k + 1) * B], ridx)
            assert np.array_equal(_np(prio)[k * B:(k + 1) * B], rprio)
            rw = OR.is_weights(rprio, ref.root, rp.top, 0.6)
            np.testing.assert_allclose(_np(w)[k * B:(k + 1) * B], rw, rtol=1e-5)
        assert (_np(prio) > 0).all()
    # priority update with duplicates (last writer wins), evicted leaves skipped, max_p tracking
    ids = rng.randint(0, N, 700).astype(np.int64)
    ids[100:110] = ids[0]
    loss = (np.abs(rng.randn(700)) * 3).astype(np.float32)
    rp.update_priority(torch.as_tensor(ids), torch.as_tensor(loss))
    newp = new_priority(loss, 0.01, 0.5)
    keep = ref.leaves()[ids] > 0
    ref.set(ids[keep], newp[keep])
    assert np.array_equal(_np(rp.tree)[:2 * ref.P], ref.nodes)
    assert rp.max_p == pytest.approx(max(1.0, float(loss.max())), rel=1e-7)
    # the law: empirical draw frequencies follow p_i / sum p (the reference's multinomial law)
    counts = np.zeros(N)
    for _ in range(40):
        b = rp.sample(512, k_batches=4)
        np.add.at(counts, _np(b.indices), 1)
    law = ref.leaves().astype(np.float64); law /= law.sum()
    assert np.corrcoef(counts / counts.sum(), law)[0, 1] > 0.95


def test_sampler_own_generator_matches_oracle_philox_and_advances_per_launch():
    """a0_pt_sample_rng: uniforms bit-equal to oracle.sumtree.philox_uniform(seed, call, n), indices
    equal to the oracle sum-tree fed those uniforms; the device-resident call counter advances with
    every launch and every replay of a captured graph; rng_seek repositions it."""
    from oracle.sumtree import philox_uniform
    N, Bn, k = 4096, 32, 5
    rp = _replay(N, per=True, native=True, E=4)
    from agent0_b200.synth import fill_shard_synthetic
    fill_shard_synthetic(rp, N, 4, 1)
    ids = torch.arange(0, rp.top, 3, device="cuda")
    rp.update_priority(ids, torch.rand(len(ids), device="cuda", generator=torch.Generator("cuda").manual_seed(2)) * 5)
    tree = SumTree(N)
    tree.set(np.arange(N), _np(rp.priority.leaves()))
    total = Bn * k
    u_out = torch.empty(total, device="cuda")
    seed = 0x1234_5678_9ABC_DEF0

    def check(call, batch):
        want_u = philox_uniform(seed, call, total)
        assert np.array_equal(_np(u_out), want_u)
        want_idx = np.concatenate([tree.sample_stratified(want_u[j * Bn:(j + 1) * Bn])[0] for j in range(k)])
        assert np.array_equal(_np(batch.indices), want_idx)

    check(7, rp.sample(Bn, k_batches=k, seed=seed, call=7, u_out=u_out))           # explicit call number
    for call in (0, 1, 2):                                                             # device counter: 0, 1, 2, ...
        check(call, rp.sample(Bn, k_batches=k, seed=seed, u_out=u_out))
    rp.rng_seek(2 ** 33 + 5)                                                           # 64-bit call numbers
    check(2 ** 33 + 5, rp.sample(Bn, k_batches=k, seed=seed, u_out=u_out))
    # captured graph: every replay draws the next call
    out = rp.alloc_batch(total)
    rp.push_dynamic()
    rp.rng_seek(100)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        rp.sample(Bn, k_batches=k, seed=seed, u_out=u_out, out=out, dynamic=True)
    for call in (100, 101, 102):
        g.replay()
        torch.cuda.synchronize()
        check(call, out)


@pytest.mark.parametrize("per,Bn", [(True, 12), (False, 32), (False, 5)])
def test_sampler_own_generator_other_launch_shapes(per, Bn):
    """The device call counter must advance exactly once per launch on every epilogue path: batch sizes
    that are not a multiple of the warps per CTA (per-warp tickets) and the uniform policy (no weights
    epilogue, per-CTA arrivals)."""
    from oracle.sumtree import philox_uniform
    N, k = 1024, 3
    rp = _replay(N, per=per, native=True, E=4)
    from agent0_b200.synth import fill_shard_synthetic
    fill_shard_synthetic(rp, N, 4, 1)
    tree = SumTree(N)
    tree.set(np.arange(N), _np(rp.priority.leaves()))
    total = Bn * k
    u_out = torch.empty(total, device="cuda")
    for call in range(4):
        b = rp.sample(Bn, k_batches=k, seed=5, u_out=u_out)
        want_u = philox_uniform(5, call, total)
        assert np.array_equal(_np(u_out), want_u)
        want_idx = np.concatenate([tree.sample_stratified(want_u[j * Bn:(j + 1) * Bn])[0] for j in range(k)])
        assert np.array_equal(_np(b.indices), want_idx)
        if not per:
            assert bool((b.weights == 1).all())
        else:
            w = _np(b.weights).reshape(k, Bn)
            assert np.allclose(w.max(axis=1), 1.0, atol=1e-6)


@pytest.mark.parametrize("N", [2, 5, 2048, 4096, 70000, 3_000_000, 1 << 24])
def test_sumtree_update_paths_all_depths_and_sizes(N):
    """K2b at tree depths 1, 3, 11, 12, 17, 22 and 24 and at every launch shape: one CTA with the shared-memory
    node map (<= 1024 indices), a cluster of up to 8 CTAs climbing the paths, the cluster leaf write + chunk rebuild on all SMs (from 2048 indices
    with >= 4 per chunk), and the one-CTA write + rebuild above 16384 indices -- always the oracle's tree."""
    rp = _replay(N, per=True, **({"frame_capacity": 65536} if N > 1_000_000 else {}))     # 3 M leaves: depth 22, 10 sparse levels
    rng = np.random.RandomState(N)
    ref = SumTree(N)
    pr = (rng.rand(N).astype(np.float32) + 0.1)
    ref.build(pr)
    for lo in range(0, N, 30000):                      # > 16384 per call: write + rebuild kernels
        hi = min(N, lo + 30000)
        rp.set_priorities(torch.arange(lo, hi), torch.as_tensor(pr[lo:hi]))
    assert np.array_equal(_np(rp.tree)[:2 * ref.P], ref.nodes)
    for count in (1, 31, 1024, 1025, 3000, 10240, 16384, 16385):
        ids = rng.randint(0, N, count).astype(np.int64)
        if count > 8:
            ids[-3:] = ids[0]                               # duplicates: the last one wins
        loss = (np.abs(rng.randn(count)) * 2).astype(np.float32)
        rp.update_priority(torch.as_tensor(ids), torch.as_tensor(loss))
        ref.set(ids, new_priority(loss, 0.01, 0.5))
        assert np.array_equal(_np(rp.tree)[:2 * ref.P], ref.nodes), count
    assert rp.max_p >= 1.0


def test_per_bookkeeping_new_entries_beta_and_compat_sum(golden):
    """extend(): new records get max_p^alpha, beta follows LinearSchedule, IS weights follow
    trainer.py:91-94 (with the reference's all-slots denominator when compat_sum=True)."""
    g = golden("replay_n1")
    rp = _replay(256, per=True, compat_sum=True)
    assert rp.beta == 0.4
    rp.extend(_tuples(g, 0, 30))
    assert rp.beta == 0.4                                   # value before advancing (replay.py:53)
    leaves = _np(rp.priority.leaves())
    assert (leaves[:30] == 1.0).all() and (leaves[30:] == 0).all()
    loss = np.linspace(0.5, 9.0, 30).astype(np.float32)
    rp.update_priority(torch.arange(30), torch.as_tensor(loss))
    rp.extend(_tuples(g, 30, 50))
    assert rp.beta == pytest.approx(0.4 + 0.6 / 1000 * 30)
    leaves = _np(rp.priority.leaves())
    np.testing.assert_allclose(leaves[:30], new_priority(loss, 0.01, 0.5), rtol=1e-6)
    np.testing.assert_allclose(leaves[30:50], np.sqrt(np.float32(9.0)), rtol=1e-6)    # max_p ** alpha
    u = torch.rand(8, device="cuda")
    b = rp.sample(8, u=u)
    sum_all = leaves.sum() + (256 - 50)                     # never-written slots hold 1.0 (SURVEY Q3)
    w = OR.is_weights(_np(b.priorities), sum_all, 50, rp.beta)
    np.testing.assert_allclose(_np(b.weights), w, rtol=1e-5)
    assert np.array_equal(_np(b.priorities), leaves[_np(b.indices)])


def test_uniform_policy_weights_are_one(golden):
    g = golden("replay_n1")
    rp = _replay(256, per=False)
    rp.extend(_tuples(g, 0, 60))
    b = rp.sample(16, k_batches=2)
    assert (_np(b.weights) == 1.0).all() and (_np(b.priorities) == 1.0).all()
    assert _np(b.indices).max() < 60
    rp.update_priority(b.indices, torch.rand(32))           # no-op for uniform replay
    assert (_np(rp.priority.leaves())[:60] == 1.0).all()


def test_trainer_step_golden_weights_and_priorities(golden):
    """The reference's real Trainer.step (C51, PER, n=3): same indices -> same batch fields, IS
    weights and priorities after update_priority."""
    g = golden("trainer_step")
    s = record_stream(int(g["num_envs"]), int(g["steps"]), seed=int(g["seed"]), p_terminal=0.05,
                      p_life_loss=0.05, p_truncated=0.03)
    fr, a, r, d = OR.pack_nstep(s["obs"], s["action"], s["reward"], s["done"], int(g["n_step"]), 0.99)
    # the reference deque (maxlen 64) dropped the oldest 26 of the 90 entries
    drop = len(a) - 64
    rp = _replay(64, per=True, compat_sum=True, frame_capacity=2048)
    rp.extend([(fr[i].tobytes(), a[i], r[i], d[i]) for i in range(drop, len(a))])
    assert rp.top == int(g["top"])
    for it in range(len(g["batches"])):
        idx = g["batches"][it] % rp.top
        b = rp.sample(8, indices=torch.as_tensor(idx))
        np.testing.assert_allclose(_np(b.weights), g["weights"][it], rtol=1e-5)
        assert np.array_equal(_np(b.rewards_f32), g["rewards"][it])
        assert np.array_equal(_np(b.terminals_f32), g["dones"][it])
        assert np.array_equal(_np(b.actions).astype(np.float32), g["actions"][it])
        assert np.array_equal(_np(b.frames).astype(np.uint64).sum(axis=1), g["frames_crc"][it])
        rp.update_priority(b.indices, torch.as_tensor(g["q_loss"][it]))
        np.testing.assert_allclose(_np(rp.priority.leaves()), g["prio_after"][it], rtol=1e-5)
        assert rp.max_p == pytest.approx(float(g["max_p_after"][it]), rel=1e-6)


def test_empty_and_error_paths():
    from agent0_b200 import _lib
    rp = _replay(64)
    rp.extend([])
    with pytest.raises(RuntimeError):
        rp.sample(4)
    lib = _lib.load()
    assert lib.a0_rb_gather(rp.h, None, 4, 1, 0.99, None, None, None, None, None, None, None, 0, None) != 0
    assert b"required" in lib.a0_last_error()
    assert lib.a0_rb_gather(rp.h, None, 0, 1, 0.99, None, None, None, None, None, None, None, 0, None) == 0


@pytest.mark.parametrize("n", [1, 3])
def test_fused_bf16_gather_equals_torch_cast_of_the_f32_gather(golden, n):
    """a0_rb_gather_bf16 (mixed-precision learner input, SURVEY 8f-2): every value is
    bf16(fl32(norm(x))) rounded to nearest even -- bit-identical to casting the f32 gather with torch,
    for all 256 byte values and the three normalisations, on the golden actor stream (n-step window,
    episode boundaries) and into preallocated out= buffers; scalars as the f32 gather."""
    from agent0_b200.replay import NORM_RECIP
    E = 2
    rp = _replay(64, n=1, native=True, E=E)
    ramp = (np.arange(4 * 84 * 84, dtype=np.int64) % 256).astype(np.uint8).reshape(4, 84, 84)
    rp.reset_streams(np.arange(E), np.stack([ramp, ramp[::-1].copy()]))
    new = np.stack([np.full((84, 84), 255, np.uint8), np.zeros((84, 84), np.uint8)])
    rp.append_steps(np.arange(E), np.ones(E, dtype=np.int64), new, np.array([1, 2]), np.array([0.5, -1.0]), np.array([False, True]))
    pos = torch.arange(E, device="cuda")
    for mode in (0, 1, 2):
        f = rp.gather(pos, normalized=mode)
        h = rp.gather(pos, normalized=mode, obs_dtype=torch.bfloat16)
        assert h.obs.dtype == torch.bfloat16 and h.obs.shape == f.obs.shape
        assert torch.equal(h.obs, f.obs.to(torch.bfloat16)) and torch.equal(h.next_obs, f.next_obs.to(torch.bfloat16))
        assert torch.equal(h.rewards, f.rewards) and torch.equal(h.actions, f.actions)
    out = rp.alloc_batch(E, normalized=NORM_RECIP, obs_dtype=torch.bfloat16)
    b = rp.sample(E, indices=pos, out=out, normalized=NORM_RECIP)
    assert b.obs.data_ptr() == out.obs.data_ptr()
    assert torch.equal(out.obs, rp.gather(pos, normalized=NORM_RECIP).obs.to(torch.bfloat16))
    # the golden actor stream through the native n-step path
    g = golden(f"replay_n{n}")
    E2, T = int(g["num_envs"]), int(g["steps"])
    s_obs = g["stream_obs"]
    done = OR.done_rule(g["stream_terminal"], g["stream_life_loss"], g["stream_truncated"])
    rp = _replay(256, n=n, native=True, E=E2)
    for k in range(T):
        rp.append_vector_step(s_obs[k], g["stream_action"][k], g["stream_reward"][k], done[k], s_obs[k + 1])
    live = torch.nonzero(rp.priority.leaves() > 0).view(-1)
    f = rp.gather(live, normalized=0)
    h = rp.gather(live, obs_dtype=torch.bfloat16)
    assert torch.equal(h.obs, f.obs.to(torch.bfloat16)) and torch.equal(h.next_obs, f.next_obs.to(torch.bfloat16))
    assert torch.equal(h.rewards, f.rewards) and torch.equal(h.terminals, f.terminals) and torch.equal(h.boot_indices, f.boot_indices)
