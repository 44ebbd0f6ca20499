"""K5 (a0_act_epsilon_greedy, a0_u8_to_f32) and ActorPolicy at every shape the C ABI accepts, against torch's CPU rule.

a0_act_epsilon_greedy is called directly, every output poisoned first and followed by a canary, and checked against
  * the action of oracle.reference_replay.act_rule's rule for the given draws: np.where(u > epsilon, argmax, random),
    where the arg-max is qt.max(dim=-1)'s (NaN above every number, the first index among equal values and among NaNs);
  * qmax_out equal to torch.max(q, dim=-1).values on the CPU bit for bit, NaN where torch has NaN;
  * the mean within (ceil(E/128) + 16) * 2^-24 * mean|m| of the float64 mean of those maxima, NaN where it is NaN.
Every A from 1 to 32 (a lane stands for an action), env counts on both sides of a CTA of four envs and of the
reducing CTA's 128 threads, and the 8-byte ticket reused across launches of different grid sizes and on two streams.
a0_u8_to_f32 is checked past the end of its grid-stride loop's first pass."""
import numpy as np
import pytest
import torch

from agent0_b200.config import make_config
from oracle import reference_replay as OR
from tests.frame_cases import SIZES
from tests.test_gpu_actor import _TableNet
from tests.test_gpu_replay import _norm_ref

pytestmark = pytest.mark.gpu

f32 = np.float32
ES = [1, 3, 4, 5, 127, 128, 129, 1000, 4097, 65537]
POISON = 0x7FBADBAD                       # a NaN no kernel computes: an unwritten float32 shows up in a bit compare
I64_POISON = -0x5EADBEEF
ONE_PASS = 148 * 8 * 256 * 16             # bytes a0_u8_to_f32 converts before its grid-stride loop comes round


@pytest.fixture(scope="module")
def lib():
    from agent0_b200 import _lib
    return _lib.load()


def _nan():
    return f32(np.nan)


def edge_rows(A, with_nan):
    """Rows of A values that decide the arg-max at its edges; each only where A leaves room for it."""
    inf, big, sub = f32(np.inf), f32(3.4e38), f32(1e-45)
    rows = []

    def add(cond, vals):
        if cond:
            r = np.full(A, -5.0, f32)
            r[:len(vals)] = vals
            rows.append(r)
    if not with_nan:
        add(A >= 3, [2.0, 7.0, 7.0])                      # a tie: the first index wins
        add(A >= 1, np.full(A, 1.25, f32))                # all equal
        add(A >= 2, [-0.0, 0.0])                          # +0 / -0 tie: index 0, value -0
        add(A >= 2, [0.0, -0.0])
        add(A >= 1, np.full(A, -inf, f32))                # all -inf: index 0
        add(A >= 4, [1.0, inf, 3.0, inf])                 # +inf, twice
        add(A >= 2, [-inf, inf])                          # +inf next to -inf
        add(A >= 2, [inf, -inf])
        add(A >= 3, [big, -big, big])                     # the largest finite values, tied
        add(A >= 1, np.full(A, -big, f32))
        add(A >= 3, [sub, 2 * sub, -sub])                 # subnormals
        add(A >= 2, [0.0, sub])
        add(A >= 2, [-sub, -0.0])
        r = np.linspace(-3.0, 3.0, A, dtype=f32)[::-1].copy()
        rows += [r, r.copy()]                             # identical rows
    else:
        n = _nan()
        add(A >= 1, [n])                                  # NaN first
        add(A >= 3, np.where(np.arange(A) == A // 2, n, np.arange(A, dtype=f32)))    # ... in the middle, before the largest number
        add(A >= 2, np.where(np.arange(A) == A - 1, n, np.arange(A, dtype=f32)))     # ... last
        add(A >= 4, [1.0, n, 5.0, 9.0])                   # the row a '>' butterfly split three ways
        add(A >= 1, np.full(A, n, f32))                   # all NaN
        add(A >= 2, [inf, n])                             # NaN next to +inf
        add(A >= 2, [n, inf])
        add(A >= 3, [-inf, n, n])
    return rows


def _q(rng, E, A, rows, start):
    """E rows: edge rows from index ``start`` (cycling), then random rows with some ties."""
    q = (rng.randn(E, A) * 3).astype(f32)
    q[1::5] = np.round(q[1::5])
    k = min(E, len(rows))
    for i in range(k):
        q[i] = rows[(start + i) % len(rows)]
    return q, k


def _draws(rng, E, A, eps):
    """u and action_random with the edges of the draw: u == eps (random action), u = 0 (random at eps = 0), the next
    double above eps (greedy), and random actions >= A, which pass through."""
    u = rng.rand(E)
    u[0::7] = eps
    u[3::11] = np.nextafter(eps, 1.0)
    u[5::13] = 0.0
    ar = rng.randint(0, A + 7, E).astype(np.int64)
    ar[2::9] = 2 ** 40 + 3
    return u, ar


def _expect(q, u, ar, eps):
    t = torch.from_numpy(q)
    mx, ix = torch.max(t, dim=-1)
    assert np.array_equal(ix.numpy(), q.argmax(-1)), "torch's and numpy's arg-max disagree"
    action = np.where(u > eps, ix.numpy(), ar).astype(np.int64)
    return action, mx.numpy()


def _act(lib, q, u, ar, eps, scratch, with_qmax=True, stream=None):
    """One launch into poisoned buffers with one canary element each (checked here).  Returns (rc, action,
    qmax_out or None, mean)."""
    from agent0_b200 import _lib
    E, A = q.shape
    qg = torch.from_numpy(q).cuda()
    ug = torch.from_numpy(u).cuda()
    ag = torch.from_numpy(ar).cuda()
    act = torch.full((E + 1,), I64_POISON, dtype=torch.int64, device="cuda")
    qm = torch.full((E + 1,), POISON, dtype=torch.int32, device="cuda")
    mean = torch.full((1,), POISON, dtype=torch.int32, device="cuda")
    st = stream.cuda_stream if stream is not None else _lib.stream_ptr()
    rc = lib.a0_act_epsilon_greedy(qg.data_ptr(), E, A, eps, ug.data_ptr(), ag.data_ptr(), act.data_ptr(),
                                   qm.data_ptr() if with_qmax else None, scratch.data_ptr(), mean.data_ptr(), st)
    torch.cuda.synchronize()
    act, qm, mean = act.cpu().numpy(), qm.cpu().numpy(), mean.cpu().numpy()
    assert act[E] == I64_POISON, "a0_act_epsilon_greedy wrote past action_out[E-1]"
    assert qm[E] == POISON and (with_qmax or (qm == POISON).all()), "qmax_out written where it must not be"
    return rc, act[:E], qm[:E].view(f32) if with_qmax else None, mean.view(f32)[0]


def _check_mean(tag, got, m):
    """The float64 mean of the maxima m: NaN and infinities exactly, otherwise the bound of the module docstring."""
    E = len(m)
    ref = np.mean(m.astype(np.float64))
    if not np.isfinite(ref) or not np.isfinite(m).all():
        want = f32(m.astype(np.float64).sum() / E)
        assert (np.isnan(got) and np.isnan(want)) or got == want, f"{tag}: mean {got!r}, reference {want!r}"
        return
    bound = (-(-E // 128) + 16) * 2.0 ** -24 * np.mean(np.abs(m.astype(np.float64)))
    assert abs(float(got) - ref) <= bound, f"{tag}: mean {got!r} vs float64 {ref!r}, bound {bound:.3g}"


def _run_case(lib, scratch, rng, E, A, rows, start, eps, check_mean=True):
    tag = f"E={E} A={A} eps={eps} rows {start}.."
    q, k = _q(rng, E, A, rows, start)
    u, ar = _draws(rng, E, A, eps)
    want_a, want_m = _expect(q, u, ar, eps)
    rc, act, qm, mean = _act(lib, q, u, ar, eps, scratch)
    assert rc == 0, tag
    bad = np.flatnonzero(act != want_a)
    assert bad.size == 0, f"{tag}: action of env {bad[0]} (q {q[bad[0]]!r}, u {u[bad[0]]!r}): {act[bad[0]]} != {want_a[bad[0]]}"
    bad = np.flatnonzero(qm.view(np.uint32) != want_m.view(np.uint32))
    assert bad.size == 0, f"{tag}: qmax_out of env {bad[0]} (q {q[bad[0]]!r}): {qm[bad[0]]!r} != {want_m[bad[0]]!r}"
    if check_mean:
        _check_mean(tag, mean, want_m)
    # without qmax_out: the same actions and the same mean
    rc, act2, _, mean2 = _act(lib, q, u, ar, eps, scratch, with_qmax=False)
    assert rc == 0 and np.array_equal(act2, act), f"{tag}: actions differ without qmax_out"
    assert np.array_equal(np.array([mean2]).view(np.uint32), np.array([mean]).view(np.uint32)), f"{tag}: mean differs without qmax_out"
    return k


def _scratch():
    return torch.zeros(2, dtype=torch.float32, device="cuda")


@pytest.mark.parametrize("E", ES)
def test_act_every_action_count_and_edge_row(lib, E):
    """Every A in 1..32 with ties, +-0, +-inf, -inf rows, +-3.4e38, subnormals and identical rows; the draws' edges
    and epsilon 0, 1 and between; the mean of finite maxima against its float64 bound."""
    rng = np.random.RandomState(E)
    scratch = _scratch()
    for A in range(1, 33):
        rows = edge_rows(A, with_nan=False)
        start = 0
        while start < len(rows):                  # small E: the edge rows over several launches
            start += _run_case(lib, scratch, rng, E, A, rows, start, 0.0)
        _run_case(lib, scratch, rng, E, A, rows, 0, 1.0)
        # rows whose maxima are finite: the mean against its float64 bound
        _run_case(lib, scratch, rng, E, A, [r for r in rows if np.isfinite(r.max())], 0, 0.3)
    assert not scratch.cpu().numpy().view(np.uint32).any(), "the ticket was not re-armed"


@pytest.mark.parametrize("E", ES)
def test_act_nan_rows_follow_torch_max(lib, E):
    """Rows with NaN at the first, a middle and the last index, all NaN, and NaN beside +inf: the action is the first
    NaN, qmax_out is that NaN, and the mean is NaN (torch's qt.max(dim=-1) and qt_max.mean())."""
    rng = np.random.RandomState(E + 7)
    scratch = _scratch()
    for A in range(1, 33):
        rows = edge_rows(A, with_nan=True)
        start = 0
        while start < len(rows):
            start += _run_case(lib, scratch, rng, E, A, rows, start, 0.0 if start % 2 else 0.25)
    # one NaN row among many finite ones at the largest E: the mean is NaN, not the mean of the others
    q = (rng.randn(E, 18) * 3).astype(f32)
    q[E // 2, 17] = np.nan
    u, ar = _draws(rng, E, 18, 0.0)
    want_a, want_m = _expect(q, u, ar, 0.0)
    rc, act, qm, mean = _act(lib, q, u, ar, 0.0, scratch)
    assert rc == 0 and np.isnan(mean) and np.isnan(qm[E // 2]) and want_a[E // 2] in (17, ar[E // 2])
    assert np.array_equal(act, want_a) and np.array_equal(qm.view(np.uint32), want_m.view(np.uint32))


def test_act_ticket_across_grid_sizes_and_streams(lib):
    """50 launches back to back on one scratch, E varying across CTA counts (and an E = 0 call): each result is right
    and identical launches give identical bits; then two streams, each with its own scratch, at the same time."""
    rng = np.random.RandomState(5)
    scratch = _scratch()
    sizes = [1, 4097, 5, 0, 128, 129, 65537, 3, 1000, 4, 127]
    first = {}
    for k in range(50):
        E = sizes[k % len(sizes)]
        A = 1 + (k * 7) % 32
        if E == 0:
            assert lib.a0_act_epsilon_greedy(None, 0, A, 0.5, None, None, None, None, scratch.data_ptr(), None, 0) == 0
            continue
        r = np.random.RandomState(1000 * E + A)       # the same inputs each time this (E, A) comes round
        q = (r.randn(E, A) * 3).astype(f32)
        u, ar = _draws(r, E, A, 0.25)
        want_a, want_m = _expect(q, u, ar, 0.25)
        rc, act, qm, mean = _act(lib, q, u, ar, 0.25, scratch)
        assert rc == 0 and np.array_equal(act, want_a) and np.array_equal(qm.view(np.uint32), want_m.view(np.uint32)), f"launch {k}"
        _check_mean(f"launch {k} E={E} A={A}", mean, want_m)
        bits = (act.tobytes(), qm.tobytes(), np.float32(mean).tobytes())
        assert first.setdefault((E, A), bits) == bits, f"launch {k}: E={E} A={A} differs from its first launch"
    assert not scratch.cpu().numpy().view(np.uint32).any(), "the ticket was not re-armed"
    # two streams, each with its own scratch, launched back to back before either is waited for
    from agent0_b200 import _lib
    E, A = 65537, 18
    q = (rng.randn(2, E, A) * 3).astype(f32)
    draws = [_draws(rng, E, A, 0.1) for _ in range(2)]
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    scr = [_scratch(), _scratch()]
    ins = [tuple(torch.from_numpy(x).cuda() for x in (q[s], draws[s][0], draws[s][1])) for s in range(2)]
    outs = [(torch.full((E,), I64_POISON, dtype=torch.int64, device="cuda"), torch.full((1,), POISON, dtype=torch.int32, device="cuda"))
            for _ in range(2)]
    torch.cuda.synchronize()
    for rep in range(8):
        for s in range(2):
            qg, ug, ag = ins[s]
            _lib.check(lib.a0_act_epsilon_greedy(qg.data_ptr(), E, A, 0.1, ug.data_ptr(), ag.data_ptr(), outs[s][0].data_ptr(), None,
                                                 scr[s].data_ptr(), outs[s][1].data_ptr(), streams[s].cuda_stream), "a0_act_epsilon_greedy")
    torch.cuda.synchronize()
    for s in range(2):
        want_a, want_m = _expect(q[s], draws[s][0], draws[s][1], 0.1)
        assert np.array_equal(outs[s][0].cpu().numpy(), want_a), f"stream {s}: actions"
        _check_mean(f"stream {s}", outs[s][1].cpu().numpy().view(f32)[0], want_m)
        assert not scr[s].cpu().numpy().view(np.uint32).any(), f"stream {s}: the ticket was not re-armed"


def test_act_empty_and_argument_errors(lib):
    """E = 0 returns 0 and writes nothing; A = 0, A = 33, E < 0 and NULL arguments are refused with a message."""
    from agent0_b200 import _lib
    E, A = 8, 4
    q = torch.randn(E, A, device="cuda")
    u = torch.rand(E, dtype=torch.float64, device="cuda")
    ar = torch.zeros(E, dtype=torch.int64, device="cuda")
    act = torch.full((E,), I64_POISON, dtype=torch.int64, device="cuda")
    qm = torch.full((E,), POISON, dtype=torch.int32, device="cuda")
    mean = torch.full((1,), POISON, dtype=torch.int32, device="cuda")
    scratch = _scratch()
    st = _lib.stream_ptr()
    args = [q.data_ptr(), E, A, 0.5, u.data_ptr(), ar.data_ptr(), act.data_ptr(), qm.data_ptr(), scratch.data_ptr(), mean.data_ptr(), st]
    assert lib.a0_act_epsilon_greedy(*(args[:1] + [0] + args[2:])) == 0
    torch.cuda.synchronize()
    assert (act == I64_POISON).all() and (qm == POISON).all() and (mean == POISON).all() and not scratch.any()

    def refused(i, v, words):
        a = list(args)
        a[i] = v
        assert lib.a0_act_epsilon_greedy(*a) == -1, (i, v)
        msg = lib.a0_last_error().decode()
        assert all(w in msg for w in words), msg
    refused(2, 0, ["action_dim 0 outside [1,32]"])
    refused(2, 33, ["action_dim 33 outside [1,32]"])
    refused(1, -1, ["negative env count"])
    for i in (0, 4, 5, 6, 8, 9):
        refused(i, None, ["NULL argument"])
    torch.cuda.synchronize()
    assert (act == I64_POISON).all() and (mean == POISON).all() and not scratch.any()


# ---------------------------------------------------------------------------------------------------- a0_u8_to_f32
COUNTS = [16, 16 * 255, 16 * 256, 16 * 257, ONE_PASS - 16, ONE_PASS, ONE_PASS + 16, 3 * ONE_PASS + 48, 256 * 4 * 84 * 84]


@pytest.mark.parametrize("count", COUNTS)
def test_u8_to_f32_counts(lib, count):
    """All three modes bit for bit against the host restatement, mode 1 against torch's CUDA .float().div(255), the
    canary after ``count`` untouched, and pointers 16 bytes into their buffers accepted."""
    from agent0_b200 import _lib
    rng = np.random.RandomState(count % 9973)
    x = rng.randint(0, 256, count + 32, dtype=np.uint8)
    x[:256] = np.arange(256, dtype=np.uint8)[:len(x)]         # every byte value
    xg = torch.from_numpy(x).cuda()
    for mode in (0, 1, 2):
        for off in (0, 16):
            out = torch.full((count + 8,), POISON, dtype=torch.int32, device="cuda")
            _lib.check(lib.a0_u8_to_f32(xg.data_ptr() + off, out.data_ptr() + off, count, mode, _lib.stream_ptr()), "a0_u8_to_f32")
            o = out.cpu().numpy()
            lo = off // 4                                  # the output pointer was 16 bytes = 4 floats in
            got = o[lo:lo + count].view(f32)
            want = _norm_ref(x[off:off + count], mode)
            bad = np.flatnonzero(got.view(np.uint32) != want.view(np.uint32))
            assert bad.size == 0, f"count={count} mode={mode} offset={off}: element {bad[0]}: {got[bad[0]]!r} != {want[bad[0]]!r}"
            assert (o[:lo] == POISON).all() and (o[lo + count:] == POISON).all(), f"count={count} mode={mode}: written outside"
            if mode == 1 and off == 0:
                assert torch.equal(out[:count].view(torch.float32), xg[:count].float().div(255.0)), f"count={count}: mode 1 vs torch"


def test_u8_to_f32_refuses_misaligned_pointers(lib):
    from agent0_b200 import _lib
    x = torch.zeros(64, dtype=torch.uint8, device="cuda")
    out = torch.full((64,), POISON, dtype=torch.int32, device="cuda")
    for pin, pout in ((8, 0), (0, 4), (8, 4)):
        assert lib.a0_u8_to_f32(x.data_ptr() + pin, out.data_ptr() + pout, 32, 0, _lib.stream_ptr()) == -1
        assert "pointers must be 16-byte aligned" in lib.a0_last_error().decode()
    torch.cuda.synchronize()
    assert (out == POISON).all()


# ---------------------------------------------------------------------------------------------------- ActorPolicy
FRAMES = [s for s, _ in SIZES if int(np.prod(s)) in (16, 7056, 25600)]


@pytest.mark.parametrize("A", [1, 18, 32])
@pytest.mark.parametrize("mode", [0, 1], ids=["NORM_DIV", "NORM_RECIP"])
def test_actor_policy_shapes(A, mode):
    """ActorPolicy.act at E in {1, 3, 256} and three frame sizes, one policy for all of them (the same E comes back with
    another frame shape): the network sees the host conversion bit for bit, the actions are act_rule's for the same
    RandomState, the mean is within the bound.  E = 256 at 84 x 84 runs the conversion's grid-stride loop."""
    from agent0_b200.actor import ActorPolicy
    from agent0_b200.replay import NORM_DIV, NORM_RECIP
    norm = (NORM_DIV, NORM_RECIP)[mode]
    assert norm == mode
    net = _TableNet(np.zeros((1, A), f32))
    pol = ActorPolicy(make_config("dqn", action_dim=A), net, norm_mode=norm, rng=np.random.RandomState(A))
    ref_rng = np.random.RandomState(A)
    rng = np.random.RandomState(100 + A + mode)
    for E in (1, 3, 256):
        for shape in FRAMES:
            obs = rng.randint(0, 256, (E, 4) + tuple(shape)).astype(np.uint8)
            q = (rng.randn(E, A) * 3).astype(f32)
            q[::4] = np.round(q[::4])                               # ties
            net.q = torch.from_numpy(q).cuda()
            for eps in (0.0, 0.5, 1.0):
                tag = f"E={E} frame={shape} eps={eps}"
                a, m = pol.act(obs, eps)
                assert np.array_equal(net.seen.cpu().numpy().view(np.uint32), _norm_ref(obs, mode).view(np.uint32)), tag
                want, _ = OR.act_rule(q, eps, A, rng=ref_rng)
                assert a.dtype == np.int64 and np.array_equal(a, want), tag
                _check_mean(tag, f32(m), q.max(-1))
