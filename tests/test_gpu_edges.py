"""Edge cases of the C ABI on the GPU: limits (n_step 16, 32 actions, 128 atoms, 256 quantiles),
other frame sizes, static screens (0 new frames per step), ragged and empty calls, argument
errors, stale priority updates after eviction, and the library options."""
import ctypes as C

import numpy as np
import pytest
import torch

from agent0_b200 import _lib
from agent0_b200.config import make_config
from oracle import losses as OL
from oracle import reference_replay as OR
from tests import parity

pytestmark = pytest.mark.gpu


def _np(t):
    return t.detach().cpu().numpy()


def _replay(size, n, E, obs_hw=(84, 84), **kw):
    from agent0_b200.replay import ReplayDataset
    cfg = make_config("dqn", per=True, n_step=n, batch_size=8, replay_size=size, num_envs=E)
    cfg.obs_shape = (4,) + tuple(obs_hw)
    return ReplayDataset(cfg, native_nstep=True, **kw)


def _stream(E, T, hw, seed, p_new4=0.1, p_static=0.0):
    """obs[k] u8[E,4,h,w]; ordinary step shifts by one new frame, p_new4: whole new stack,
    p_static: nothing changes (n_new = 0, a paused screen)."""
    rng = np.random.RandomState(seed)
    shape = tuple(hw)                      # any frame shape: (h, w), (h, w, c)
    obs = [rng.randint(0, 256, (E, 4) + shape).astype(np.uint8)]
    n_new = []
    for k in range(T):
        cur = obs[-1].copy()
        kk = np.ones(E, dtype=np.int64)
        r = rng.rand(E)
        kk[r < p_new4] = 4
        kk[(r >= p_new4) & (r < p_new4 + p_static)] = 0
        for e in range(E):
            if kk[e] == 4:
                cur[e] = rng.randint(0, 256, (4,) + shape)
            elif kk[e] == 1:
                cur[e, :3] = obs[-1][e, 1:]
                cur[e, 3] = rng.randint(0, 256, shape)
        obs.append(cur)
        n_new.append(kk)
    act = rng.randint(0, 18, (T, E)).astype(np.int64)
    rew = rng.randn(T, E)
    done = rng.rand(T, E) < 0.15
    return np.stack(obs), np.stack(n_new), act, rew, done


@pytest.mark.parametrize("n,hw,p_static", [(16, (84, 84), 0.0), (5, (96, 96), 0.3), (2, (16, 16), 0.5), (1, (84, 84), 0.2)])
def test_nstep_limits_frame_sizes_and_static_screens(n, hw, p_static):
    """K1/K3 against the oracle's actor packer for n up to A0_MAX_NSTEP, frames of 96x96 and 16x16
    bytes, and streams whose screen does not change (0 new frames: stacks share all four slots)."""
    E, T = 3, 60
    obs, n_new, act, rew, done = _stream(E, T, hw, seed=n, p_static=p_static)
    fr_ref, a_ref, r_ref, d_ref = OR.pack_nstep(obs, act, rew, done, n, 0.97)
    rp = _replay(512, n, E, hw)
    rp.gamma = 0.97
    rp.reset_streams(np.arange(E), obs[0])
    for k in range(T):
        new = [obs[k + 1][e, 4 - n_new[k][e]:] for e in range(E) if n_new[k][e]]
        new = np.concatenate(new) if new else np.zeros((0,) + hw, np.uint8)
        rp.append_steps(np.arange(E), n_new[k], new, act[k], rew[k], done[k])
    assert rp.top == (T - n + 1) * E
    ks, es = np.meshgrid(np.arange(n - 1, T), np.arange(E), indexing="ij")
    pos = ((ks - n + 1) * E + es).reshape(-1)
    ref_i = (ks * E + es).reshape(-1)
    for variant in (0, 1, 2, 3):
        rp.gather_variant = variant
        b = rp.gather(torch.as_tensor(pos, device="cuda"))
        assert np.array_equal(_np(b.frames), fr_ref[ref_i])
        assert np.array_equal(_np(b.rewards).view(np.int64), r_ref[ref_i].view(np.int64))
        assert np.array_equal(_np(b.terminals), d_ref[ref_i]) and np.array_equal(_np(b.actions), a_ref[ref_i])
    assert rp.index.head_fs == 4 * E + int(n_new.sum())    # one stored frame per NEW frame: static steps store none


def test_gather_after_a_smaller_frame_shard_in_another_thread():
    """K3's shared-memory limits are attributes of the kernels for the whole process: a thread that gathers from a
    shard of 16-byte frames must not lower them under a shard of 84x84 frames another thread gathers from (a per-thread
    record of the limits did, and the other thread's next gather failed to launch)."""
    import threading
    E = 2
    obs, n_new, act, rew, done = _stream(E, 6, (84, 84), seed=9)
    fr_ref = OR.pack_nstep(obs, act, rew, done, 1, 0.99)[0]
    big = _replay(64, 1, E)
    big.reset_streams(np.arange(E), obs[0])
    for k in range(6):
        new = np.concatenate([obs[k + 1][e, 4 - n_new[k][e]:] for e in range(E) if n_new[k][e]])
        big.append_steps(np.arange(E), n_new[k], new, act[k], rew[k], done[k])
    idx = torch.arange(12, device="cuda")

    def gathers(rp):
        for variant in (0, 2, 3):
            rp.gather_variant = variant
            yield variant, _np(rp.gather(idx[:rp.top]).frames)
        yield "f32", _np(rp.gather(idx[:rp.top], normalized=2).obs)

    for _, fr in gathers(big):
        assert fr.shape[0] == 12
    err = []

    def small():
        try:
            rp = _replay(64, 1, E, (4, 4))
            o = _stream(E, 2, (4, 4), seed=1)
            rp.reset_streams(np.arange(E), o[0][0])
            rp.append_steps(np.arange(E), [1] * E, o[0][1][:, 3], [0] * E, [0.0] * E, [False] * E)
            list(gathers(rp))
        except BaseException as e:          # noqa: BLE001 (re-raised in the main thread)
            err.append(e)

    t = threading.Thread(target=small)
    t.start(); t.join()
    assert not err, err
    for variant, fr in gathers(big):
        want = fr_ref[:12] if variant != "f32" else fr_ref[:12, :4 * 7056].astype(np.float32)
        assert np.array_equal(fr.reshape(12, -1), want), variant


def test_ragged_and_empty_calls():
    rp = _replay(128, 3, 4)
    obs, n_new, act, rew, done = _stream(4, 30, (84, 84), seed=2)
    rp.reset_streams(np.arange(4), obs[0])
    # ragged: streams advance at different rates, in arbitrary interleaving, several steps per call
    order = [(0, 0), (0, 1), (0, 2), (2, 0), (1, 0), (0, 3), (2, 1), (3, 0), (1, 1), (2, 2), (2, 3), (2, 4)]
    rp.append_steps([], [], np.zeros((0, 84, 84), np.uint8), [], [], [])             # empty append is a no-op
    streams = np.array([e for e, _ in order])
    kk = np.array([n_new[k][e] for e, k in order])
    new = np.concatenate([obs[k + 1][e, 4 - n_new[k][e]:] for e, k in order])
    rp.append_steps(streams, kk, new, [act[k][e] for e, k in order], [rew[k][e] for e, k in order],
                    [done[k][e] for e, k in order])
    # stream 0 has 4 steps -> 2 sampleable, stream 2 has 5 -> 3, streams 1 and 3 too short
    assert rp.top == 2 + 3
    live = np.flatnonzero(_np(rp.priority.leaves()) > 0)
    b = rp.gather(torch.as_tensor(live, device="cuda"))
    fr_ref, a_ref, r_ref, d_ref = OR.pack_nstep(obs, act, rew, done, 3, 0.99)
    for i, p in enumerate(live):
        e, k0 = order[p]
        ref = (k0 + 2) * 4 + e
        assert np.array_equal(_np(b.frames[i]), fr_ref[ref]) and _np(b.rewards[i]).view(np.int64) == r_ref[ref].view(np.int64)
    # gather of a record whose window is incomplete is flagged, not a crash
    bad = rp.gather(torch.as_tensor([len(order) - 1], device="cuda"))
    assert int(bad.actions[0]) == -1 and int(bad.boot_indices[0]) == -1
    lib = rp.lib
    assert lib.a0_pt_update(rp.h, None, None, 0, 0.5, 0.01, None) == 0
    assert lib.a0_pt_sample(rp.h, None, 0, 8, 1.0, 0.4, 0.0, 0, None, None, None, None) == 0


@pytest.mark.parametrize("n", [2, 3, 4])
def test_speculative_window_fetch_with_wrong_and_right_stride_guesses(n):
    """K3 guesses the successor of record p as p + stride (stride measured at ingest) and fetches the
    whole n-step window in one round trip; the stored links decide.  Lockstep steps (guess right),
    steps where random streams sit out (guess wrong for their neighbours), wrap-around of the record
    ring, then lockstep again so the hint is armed when the gather runs: every sampleable record must
    still return its own stream's window."""
    E, T = 5, 70
    obs, n_new, act, rew, done = _stream(E, T, (84, 84), seed=40 + n)
    rng = np.random.RandomState(n)
    rp = _replay(160, n, E, frame_capacity=900, age_limit=64)
    rp.reset_streams(np.arange(E), obs[0])
    hist = {e: [] for e in range(E)}          # per stream: ring positions of its records, in step order
    owner = {}                                # ring position -> (stream, index into hist[stream]) of its newest record
    step_of = np.zeros(E, dtype=np.int64)
    q = 0
    for rnd in range(T + 40):
        lockstep = rnd < 10 or rnd % 3 == 0 or step_of.min() >= T - 12
        es = np.arange(E) if lockstep else np.flatnonzero(rng.rand(E) < 0.6)
        es = es[step_of[es] < T]
        if len(es) == 0:
            continue
        ks = step_of[es]
        new = [obs[k + 1][e, 4 - n_new[k][e]:] for e, k in zip(es, ks) if n_new[k][e]]
        new = np.concatenate(new) if new else np.zeros((0, 84, 84), np.uint8)
        rp.append_steps(es, [n_new[k][e] for e, k in zip(es, ks)], new, [act[k][e] for e, k in zip(es, ks)],
                        [rew[k][e] for e, k in zip(es, ks)], [done[k][e] for e, k in zip(es, ks)])
        for e in es:
            owner[q % rp.size] = (e, len(hist[e]))
            hist[e].append(q % rp.size)        # record j of stream e is its step j
            q += 1
        step_of[es] += 1
    assert q == E * T > rp.size                                  # everything appended; the record ring wrapped
    live = np.flatnonzero(_np(rp.priority.leaves()) > 0)
    assert len(live) == rp.top and rp.top > 40
    fr_ref, a_ref, r_ref, d_ref = OR.pack_nstep(obs, act, rew, done, n, 0.99)
    for variant in (0, 1):
        rp.gather_variant = variant
        b = rp.gather(torch.as_tensor(live, device="cuda"))
        fr, rw, dn, ac, boot = _np(b.frames), _np(b.rewards), _np(b.terminals), _np(b.actions), _np(b.boot_indices)
        for i, p in enumerate(live):
            e, k0 = owner[int(p)]
            ref = (k0 + n - 1) * E + e
            assert np.array_equal(fr[i], fr_ref[ref]) and rw[i].view(np.int64) == r_ref[ref].view(np.int64)
            assert dn[i] == d_ref[ref] and ac[i] == a_ref[ref]
            assert boot[i] == (hist[e][k0 + n] if k0 + n < len(hist[e]) else -1)
    bf = rp.gather(torch.as_tensor(live, device="cuda"), normalized=2)
    assert np.array_equal(_np(bf.obs).astype(np.uint8).reshape(len(live), -1), fr[:, :4 * 84 * 84])
    assert np.array_equal(_np(bf.rewards).view(np.int64), rw.view(np.int64))


def test_argument_errors_carry_messages():
    lib = _lib.load()
    h = C.c_void_p()
    assert lib.a0_rb_create(C.byref(h), (1 << 24) + 1, 1 << 20, 7056, 0) == -1 and b"2^24" in lib.a0_last_error()
    assert lib.a0_rb_create(C.byref(h), 1024, 4096, 7057, 0) == -1 and b"multiple of 16" in lib.a0_last_error()
    rp = _replay(64, 1, 2)
    idx = torch.zeros(4, dtype=torch.int64, device="cuda")
    out = torch.empty(4 * 8 * 7056, dtype=torch.uint8, device="cuda")
    assert lib.a0_rb_gather(rp.h, idx.data_ptr(), 4, 17, 0.99, out.data_ptr(), None, None, None, None, None, None, 0, None) == -1
    assert b"n_step" in lib.a0_last_error()
    assert lib.a0_rb_gather(rp.h, idx.data_ptr(), 4, 1, 0.99, out.data_ptr(), None, None, None, None, None, None, 4, None) == -1
    assert lib.a0_pt_sample(rp.h, idx.data_ptr(), 10, 4, 1.0, 0.4, 0.0, 0, idx.data_ptr(), idx.data_ptr(), None, None) == -1
    assert b"multiple of batch" in lib.a0_last_error()
    c = _lib.LossCommon(B=4, A=33)
    assert lib.a0_loss_dqn(C.byref(c), None, None, None, None, None) == -1 and b"action_dim" in lib.a0_last_error()
    assert lib.a0_set_option(99, 1) == -1
    assert lib.a0_set_option(2, 5) == -1 and lib.a0_set_option(2, 3) == 0
    # out-of-range sampled positions are flagged by K3 (action -1), never dereferenced
    b = rp.gather(torch.as_tensor([-5, 64, 1 << 40], device="cuda"))
    assert (_np(b.actions) == -1).all()


def test_stale_priority_updates_after_eviction_are_dropped():
    """update_priority for a record that was evicted between sample and update must not resurrect
    its leaf (K2b skips leaves that are 0)."""
    rp = _replay(256, 1, 2, frame_capacity=120, age_limit=16)      # the frame ring, not the record ring, evicts
    obs, n_new, act, rew, done = _stream(2, 80, (84, 84), seed=3, p_new4=0.0)
    rp.reset_streams(np.arange(2), obs[0])
    step = lambda k: rp.append_steps(np.arange(2), n_new[k], np.concatenate([obs[k + 1][e, 3:] for e in range(2)]),
                                     act[k], rew[k], done[k])
    for k in range(10):
        step(k)
    old = np.arange(20, dtype=np.int64)                            # "sampled" now: all 20 records are live
    assert (_np(rp.priority.leaves())[old] > 0).all()
    for k in range(10, 60):
        step(k)
    before = _np(rp.tree).copy()
    evicted = old[~rp.index.sampleable[old]]
    assert len(evicted) > 0 and (before[rp.P + evicted] == 0).all()
    rp.update_priority(torch.as_tensor(old), torch.full((len(old),), 7.0))
    after = _np(rp.tree)
    assert (after[rp.P + evicted] == 0).all()                      # not resurrected
    alive = old[rp.index.sampleable[old]]
    np.testing.assert_allclose(after[rp.P + alive], np.sqrt(np.float32(7.01)), rtol=1e-6)
    P = rp.P
    assert np.array_equal(after[1:P], after[2:2 * P:2] + after[3:2 * P:2])
    assert rp.max_p == pytest.approx(7.0)


@pytest.mark.parametrize("A,M", [(32, 128), (1, 2), (18, 51)])
def test_c51_limits(A, M):
    from agent0_b200 import losses as L
    rng = np.random.RandomState(A * M)
    B = 37
    a = rng.randint(0, A, B).astype(np.int64)
    r = rng.choice([-1.0, 0.0, 1.0, 9.99], B).astype(np.float32)
    d = (rng.rand(B) < 0.3).astype(np.float32)
    w = (rng.rand(B) + 0.05).astype(np.float32)
    lg, tg = [(rng.randn(B, A, M) * 2).astype(np.float32) for _ in range(2)]
    atoms = np.linspace(-10, 10, M).astype(np.float32)
    dv = lambda x: torch.as_tensor(x).cuda()
    out = L.c51_loss(dv(lg), dv(tg), dv(atoms), dv(a), dv(r), dv(d), dv(w), float(np.float32(0.99)), -10.0, 10.0,
                     want_target_prob=True)
    loss, grad, m = OL.c51(lg, tg, None, a, r, d, w, 0.99, 1, atoms, -10.0, 10.0)
    parity.close("c51.target_prob[limits]", out.target_prob, m)
    parity.close("c51.loss[limits]", out.loss, loss)
    parity.close("c51.grad[limits]", out.grad, grad)


def test_quantile_limits_256_and_1():
    from agent0_b200 import losses as L
    rng = np.random.RandomState(5)
    dv = lambda x: torch.as_tensor(x).cuda()
    for B, A, N in ((9, 32, 256), (4, 1, 1), (6, 3, 33)):
        a = rng.randint(0, A, B).astype(np.int64)
        r = rng.randn(B).astype(np.float32); d = (rng.rand(B) < 0.3).astype(np.float32); w = (rng.rand(B) + 0.1).astype(np.float32)
        q, tn = [(rng.randn(B, A, N) * 3).astype(np.float32) for _ in range(2)]
        out = L.qr_loss(dv(q), dv(tn), dv(a), dv(r), dv(d), dv(w), float(np.float32(0.99 ** 3)))
        loss, grad = OL.qr(q, tn, None, a, r, d, w, 0.99, 3)
        parity.close("quantile.loss[limits]", out.loss, loss)
        parity.close("quantile.grad[limits]", out.grad, grad)
    with pytest.raises(RuntimeError, match="outside"):
        L.qr_loss(torch.zeros(2, 2, 257).cuda(), torch.zeros(2, 2, 257).cuda(), torch.zeros(2).long().cuda(), torch.zeros(2).cuda(),
                  torch.zeros(2).cuda(), torch.ones(2).cuda(), 0.99)


def test_pdl_option_does_not_change_results():
    from agent0_b200 import losses as L
    lib = _lib.load()
    rng = np.random.RandomState(1)
    B, A, M = 64, 4, 51
    dv = lambda x: torch.as_tensor(x).cuda()
    args = (dv((rng.randn(B, A, M) * 3).astype(np.float32)), dv((rng.randn(B, A, M) * 3).astype(np.float32)),
            dv(np.linspace(-10, 10, M).astype(np.float32)), dv(rng.randint(0, A, B)), dv(rng.randn(B).astype(np.float32)),
            dv(np.zeros(B, np.float32)), dv(np.ones(B, np.float32)), 0.97, -10.0, 10.0)
    outs = []
    for mask in (0, 15, 1):
        assert lib.a0_set_option(1, mask) == 0
        outs.append([L.c51_loss(*args) for _ in range(5)][-1])
    torch.cuda.synchronize()
    assert torch.equal(outs[0].loss, outs[1].loss) and torch.equal(outs[0].grad, outs[2].grad)


def test_k2b_schedules_build_the_same_tree():
    """The K2b schedules (one CTA per chunk in a single launch / one CTA with a shared-memory node map / cluster
    path climb / cluster leaf write + chunk rebuild on all SMs / one-CTA write + rebuild) are selected by count and
    tree size; forced onto the same inputs through A0_OPT_K2B_CHUNKS, _SMALL and _BULK_MIN they must leave bit-identical trees and
    max_p, duplicates, out-of-range indices and evicted leaves included."""
    lib = _lib.load()
    N = 20000
    trees = []
    try:
        # sparse: the chunk schedule climbs up to that many updated paths per chunk one by one (A0_OPT_K2B_SPARSE), else
        # recomputes the whole chunk
        for chunks, small, bulk_min, sparse in ((1, 0, 2048, 32), (1, 0, 2048, 0), (1, 0, 2048, 3), (0, 1, 1 << 30, 32), (0, 0, 1 << 30, 32),
                                               (0, 0, 1, 32), (0, 1, 2048, 32)):
            assert lib.a0_set_option(8, chunks) == 0 and lib.a0_set_option(7, small) == 0 and lib.a0_set_option(3, bulk_min) == 0
            assert lib.a0_set_option(12, sparse) == 0
            rp = _replay(N, 1, 4)
            rp.set_priorities(torch.arange(N), torch.as_tensor((np.arange(N) % 97 + 1).astype(np.float32)))
            rp.set_priorities(torch.arange(0, N, 5), torch.zeros(N // 5))            # "evicted" leaves are skipped by updates
            r2 = np.random.RandomState(4)
            for count in (1, 40, 700, 1024, 2048, 5000, 16000):
                ids = r2.randint(0, N, count).astype(np.int64)
                if count > 8:
                    ids[-7:] = ids[3]
                    ids[5] = N + 3                                                   # out of range: ignored
                    ids[6:9] = ids[6] | 1                                            # siblings / shared parents
                rp.update_priority(torch.as_tensor(ids), torch.as_tensor(np.abs(r2.randn(count)).astype(np.float32)))
            trees.append((rp.tree.clone(), float(rp.max_p_tensor)))
            tr = trees[-1][0].cpu().numpy()
            for node in (1, 2, 77, rp.P // 2 + 5, rp.P - 1):
                assert tr[node] == np.float32(tr[2 * node] + tr[2 * node + 1])
    finally:
        lib.a0_set_option(3, 2048)
        lib.a0_set_option(7, 0)
        lib.a0_set_option(8, 1)
        lib.a0_set_option(12, 32)
    assert lib.a0_set_option(12, 33) == -1
    for t, mp in trees[1:]:
        assert torch.equal(trees[0][0], t) and trees[0][1] == mp
    assert lib.a0_set_option(3, 0) == -1


def _shard_state(rp):
    """Every piece of device state an ingest touches, as host arrays."""
    lib = _lib.load()
    dev = rp.device
    slots = _lib.device_view(lib.a0_rb_ptr(rp.h, _lib.PTR_REC_SLOTS), (rp.size, 8), "<i4", dev)
    info = _lib.device_view(lib.a0_rb_ptr(rp.h, _lib.PTR_REC_INFO), (rp.size, 4), "<i4", dev)
    scal = _lib.device_view(lib.a0_rb_ptr(rp.h, _lib.PTR_MAX_P), (19,), "<f4", dev)      # max_p, ..., dyn at [16..18]
    torch.cuda.synchronize()
    return [_np(rp.frames), _np(slots), _np(info), _np(rp.tree), _np(scal)]


@pytest.mark.parametrize("compat", [False, True])
def test_fused_ingest_launch_and_dynamic_publication_equal_the_separate_launches(compat):
    """A step-sized ingest applies marks + append (+ top/beta/sum_offset publication) in ONE launch
    (a0_k1_append_mark); with A0_OPT_FUSED_INGEST off and push_dynamic() as its own launch the shard
    must end up bit-identical: frames, records, links, the whole tree, max_p and the dyn scalars --
    on a ring smaller than the stream (evictions every step) and with n_new in {0, 1, 4}."""
    lib = _lib.load()
    E, T, n = 4, 70, 3
    obs, n_new, act, rew, done = _stream(E, T, (84, 84), seed=31, p_new4=0.1, p_static=0.1)
    states = []
    try:
        for fused in (1, 0):
            assert lib.a0_set_option(4, fused) == 0
            rp = _replay(96, n, E, frame_capacity=400, age_limit=32, compat_sum=compat)
            rp.frames.zero_()                           # cudaMalloc'd, never-written slots would differ
            rp.reset_streams(np.arange(E), obs[0])
            for k in range(T):
                new = np.concatenate([obs[k + 1][e, 4 - n_new[k][e]:] for e in range(E)]) if n_new[k].sum() else \
                    np.zeros((0, 84, 84), dtype=np.uint8)
                if k % 9 == 0:                          # some losses, so that max_p moves between appends
                    live = torch.nonzero(rp.priority.leaves() > 0).view(-1)[:5]
                    rp.update_priority(live, torch.full((len(live),), 1.5 + k, device="cuda"))
                rp.append_steps(np.arange(E), n_new[k], new, act[k], rew[k], done[k], publish_dynamic=bool(fused))
                if not fused:
                    rp.push_dynamic()
            # an empty append still publishes
            z = np.zeros(0, dtype=np.int64)
            rp.beta = 0.77
            rp.beta_schedule = lambda m: 0.77
            rp.append_steps(z, z, np.zeros((0, 84, 84), dtype=np.uint8), z, z.astype(np.float64), z.astype(bool),
                            publish_dynamic=bool(fused))
            if not fused:
                rp.push_dynamic()
            assert rp.index.tail_q > 0
            states.append(_shard_state(rp))
            assert states[-1][4][16] == float(rp.index.top) and states[-1][4][17] == np.float32(0.77)
            assert states[-1][4][18] == (float(rp.size - rp.index.top) if compat else 0.0)
    finally:
        lib.a0_set_option(4, 1)
    for a, b in zip(*states):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("A,M,B", [(4, 51, 32), (6, 64, 37), (3, 33, 5), (1, 2, 9), (5, 51, 512), (4, 32, 64)])
def test_c51_short_chain_kernel_is_bit_identical_to_the_general_kernel_and_matches_the_oracle(A, M, B):
    """a0_loss_c51 has a second kernel for the Atari shape (qsel given, A <= 6, M <= 64) whose dependent
    instruction chain is shorter (local arg-max, paired reductions, u = l + 1, read-modify-write bins,
    16-byte gradient stores).  A0_OPT_C51_FAST = 0 forces the general kernel: loss, gradient, priorities,
    projected distribution and max_p must agree bit for bit, and both with the oracle to 1e-5 -- including
    returns that clamp at the support's ends, terminal transitions (all mass to one bin), exact-integer
    bin positions, ties in the selection values, unaligned gradient blocks (A*M not a multiple of 4)."""
    from agent0_b200 import losses as L
    lib = _lib.load()
    rng = np.random.RandomState(A * M + B)
    a = rng.randint(0, A, B).astype(np.int64)
    r = rng.choice([-1.0, 0.0, 1.0, 9.99, -30.0, 30.0, 0.4, 2.0], B).astype(np.float32)
    d = (rng.rand(B) < 0.3).astype(np.float32)
    w = (rng.rand(B) + 0.05).astype(np.float32)
    lg, tg = [(rng.randn(B, A, M) * 2).astype(np.float32) for _ in range(2)]
    qs = rng.randn(B, A).astype(np.float32)
    qs[::3] = np.round(qs[::3])                       # ties: the first maximum wins
    atoms = np.linspace(-10, 10, M).astype(np.float32)
    dv = lambda x: torch.as_tensor(x).cuda()
    outs = []
    try:
        for fast in (1, 0):
            assert lib.a0_set_option(5, fast) == 0
            mp = torch.full((1,), 0.25, device="cuda")
            o = L.c51_loss(dv(lg), dv(tg), dv(atoms), dv(a), dv(r), dv(d), dv(w), float(np.float32(0.99 ** 3)), -10.0, 10.0,
                           qsel=dv(qs), want_target_prob=True, max_p=mp)
            torch.cuda.synchronize()
            outs.append((o, mp))
    finally:
        lib.a0_set_option(5, 1)
    (f, mpf), (g, mpg) = outs
    assert torch.equal(f.loss, g.loss) and torch.equal(f.grad, g.grad) and torch.equal(f.prio, g.prio)
    assert torch.equal(f.target_prob, g.target_prob) and torch.equal(mpf, mpg)
    loss, grad, m = OL.c51(lg, tg, qs, a, r, d, w, 0.99, 3, atoms, -10.0, 10.0)
    parity.close("c51.target_prob[fast kernel]", f.target_prob, m)
    parity.close("c51.loss[fast kernel]", f.loss, loss)
    parity.close("c51.grad[fast kernel]", f.grad, grad)


def test_unpaired_mailbox_gather_times_out_instead_of_hanging():
    """The gather half of a0_rb_sample_gather launched without its sampler (what a failed sampler launch or
    a mis-paired caller would leave): every CTA gives up after A0_OPT_MAIL_TIMEOUT_US, the kernel ends, the
    handle reports A0_EFAULT exactly once, and the shard keeps working."""
    import time

    from agent0_b200.replay import ReplayDataset
    from agent0_b200.synth import fill_shard_synthetic
    lib = _lib.load()
    cfg = make_config("c51", per=True, n_step=1, batch_size=8, replay_size=256, num_envs=2)
    rp = ReplayDataset(cfg, native_nstep=True)
    fill_shard_synthetic(rp, 128, 2, 3)
    out = torch.empty(8, 8 * rp.F, dtype=torch.uint8, device="cuda")
    A0_OPT_MAIL_TIMEOUT_US = 9
    _lib.check(lib.a0_set_option(A0_OPT_MAIL_TIMEOUT_US, 20000), "a0_set_option")
    try:
        t0 = time.perf_counter()
        _lib.check(lib.a0_rb_gather_unpaired(rp.h, 8, out.data_ptr(), _lib.stream_ptr(rp.device)), "a0_rb_gather_unpaired")
        torch.cuda.synchronize()
        assert time.perf_counter() - t0 < 5.0
        with pytest.raises(RuntimeError, match="timed out waiting for its sampler"):
            rp.gather(torch.arange(4, device="cuda"))
        assert lib.a0_rb_check_fault(rp.h) == 0                     # reported once, then cleared
        b = rp.sample(8, k_batches=2, seed=3)                        # the shard still works
        assert b.frames.shape[0] == 16 and int(b.indices.min()) >= 0
    finally:
        _lib.check(lib.a0_set_option(A0_OPT_MAIL_TIMEOUT_US, 2000000), "a0_set_option")


def test_views_of_shard_memory_keep_the_shard_alive():
    """replay.frames / tree / max_p_tensor are torch views of handle-owned device memory: a tensor handed to a learner
    or cached in a captured graph must keep the allocation alive after the ReplayDataset object is gone
    (a0_rb_destroy runs when the last holder of _lib.HandleOwner dies)."""
    import gc
    import weakref

    from agent0_b200.replay import ReplayDataset
    from agent0_b200.synth import fill_shard_synthetic
    cfg = make_config("c51", per=True, n_step=1, batch_size=8, replay_size=256, num_envs=2)
    rp = ReplayDataset(cfg, native_nstep=True)
    fill_shard_synthetic(rp, 128, 2, 3)
    owner = weakref.ref(rp._owner)
    max_p, leaves = rp.max_p_tensor, rp.priority.leaves()
    want = leaves.clone()
    del rp
    gc.collect()
    assert owner() is not None                              # the views hold the handle
    max_p.fill_(3.0)
    torch.cuda.synchronize()
    assert float(max_p.item()) == 3.0 and torch.equal(leaves, want)
