"""The planned priority write-back (a0_pt_update_plan + a0_pt_update_apply) against a0_pt_update_report on twin shards:
every node of the tree, max_p and the report buffers must be identical -- over tree depths 1 to 24, index counts up to
A0_K2B_PLAN_MAX, duplicates, bad losses, evicted leaves, out-of-range positions and clustered paths.  Then the captured
flagship loop (which takes the planned path at 640 indices) against the same loop forced onto the chunk schedule."""
import pytest
import torch

from agent0_b200 import _lib
from tests.test_gpu_hotloop import _outputs, _shard
from tests.test_gpu_sample_unique import RawShard, priorities

pytestmark = pytest.mark.gpu
CAP = _lib.K2B_PLAN_MAX
ALPHA, EPS = 0.5, 0.01
EINVAL = -1                  # include/agent0_b200.h: A0_EINVAL


def _twins(D, kind="spread", live_frac=1.0, N=None):
    N = N or (1 << D)
    v = priorities(kind, N, seed=D)
    if live_frac < 1.0:
        v[torch.rand(N, device="cuda", generator=torch.Generator("cuda").manual_seed(D + 1)) >= live_frac] = 0.0
    out = []
    for _ in range(2):
        sh = RawShard(N)
        assert sh.P == 1 << D
        sh.set(torch.arange(N, device="cuda"), v)
        sh.max_p = _lib.device_view(sh.lib.a0_rb_ptr(sh.h, _lib.PTR_MAX_P), (1,), "<f4", "cuda", sh.owner)
        sh.max_p.fill_(0.75)
        out.append(sh)
    torch.cuda.synchronize()
    return out


def _compare(a, b, idx, loss):
    """a: a0_pt_update_report, b: plan + apply; both with device report buffers."""
    n = idx.numel()
    rep = [(torch.full((n,), -5, dtype=torch.int64, device="cuda"), torch.full((n,), -5.0, device="cuda")) for _ in range(2)]
    st = _lib.stream_ptr()
    _lib.check(a.lib.a0_pt_update_report(a.h, idx.data_ptr(), loss.data_ptr(), n, ALPHA, EPS, rep[0][0].data_ptr(),
                                         rep[0][1].data_ptr(), st), "a0_pt_update_report")
    plan = torch.empty(_lib.K2B_PLAN_BYTES, dtype=torch.uint8, device="cuda")
    _lib.check(b.lib.a0_pt_update_plan(b.h, idx.data_ptr(), n, plan.data_ptr(), st), "a0_pt_update_plan")
    loss = loss.clone()          # the apply's predecessor on the stream writes the losses, as the last K4 does
    _lib.check(b.lib.a0_pt_update_apply(b.h, idx.data_ptr(), loss.data_ptr(), n, ALPHA, EPS, plan.data_ptr(),
                                        rep[1][0].data_ptr(), rep[1][1].data_ptr(), st), "a0_pt_update_apply")
    torch.cuda.synchronize()
    bad = (a.tree.view(torch.int32) != b.tree.view(torch.int32)).nonzero().flatten()
    assert bad.numel() == 0, f"{bad.numel()} tree nodes differ, first {bad[:8].tolist()}"
    assert torch.equal(a.max_p.view(torch.int32), b.max_p.view(torch.int32))
    assert torch.equal(rep[0][0], rep[1][0]) and torch.equal(rep[0][1].view(torch.int32), rep[1][1].view(torch.int32))


def _losses(n, seed, bad=True):
    g = torch.Generator(device="cuda").manual_seed(seed)
    loss = torch.rand(n, device="cuda", generator=g) * 3.0
    if bad and n >= 8:
        loss[1], loss[n // 2], loss[n - 3] = float("nan"), float("inf"), -0.5
    return loss


@pytest.mark.parametrize("D", [1, 3, 11, 12, 17, 20, 21, 22, 23, 24])
@pytest.mark.parametrize("count", [1, 31, 32, 33, 640, CAP])
def test_plan_apply_equals_pt_update(D, count):
    """Random positions over [-2, P + 2) on a shard of N = P - P/8 records (out-of-range on both sides and between N and
    P), NaN / infinite / negative losses, 10 % evicted leaves."""
    N = max(2, (1 << D) - (1 << D) // 8)
    a, b = _twins(D, live_frac=0.9, N=N)
    g = torch.Generator(device="cuda").manual_seed(D * 1000 + count)
    idx = torch.randint(-2, (1 << D) + 2, (count,), device="cuda", generator=g)
    _compare(a, b, idx, _losses(count, count + D))


@pytest.mark.parametrize("D", [12, 20])
@pytest.mark.parametrize("case", ["dup_nan_winner", "siblings", "one_subtree", "one_chunk", "heavy_vector", "all_evicted"])
def test_plan_apply_clustered_and_duplicate_inputs(D, case):
    kind = "heavy" if case == "heavy_vector" else "spread"
    a, b = _twins(D, kind=kind, live_frac=0.0 if case == "all_evicted" else 1.0)
    P = 1 << D
    g = torch.Generator(device="cuda").manual_seed(D)
    n = 640
    loss = _losses(n, D, bad=False)
    if case == "dup_nan_winner":                 # 20 leaves, 32 entries each; the last entry of each is the winner: NaN
        idx = torch.randint(0, P, (20,), device="cuda", generator=g).repeat(32)
        loss[-20:] = float("nan")
        loss[-40:-20] = float("inf")
    elif case == "siblings":                     # both children of 320 parents
        par = torch.randperm(P // 2, device="cuda", generator=g)[:320]
        idx = torch.stack((2 * par, 2 * par + 1), 1).flatten()
    elif case in ("one_subtree", "one_chunk"):   # every winner under one node of 1024 / 4096 leaves
        w = min(P, 1024 if case == "one_subtree" else 4096)
        base = int(torch.randint(0, P // w, (1,), generator=torch.Generator().manual_seed(D))) * w
        n = CAP if case == "one_subtree" else n
        loss = _losses(n, D)
        idx = base + (torch.randperm(w, device="cuda", generator=g)[:n] if w >= n else torch.randint(0, w, (n,), device="cuda", generator=g))
    elif case == "heavy_vector":                 # the draw of the "100 records hold 90 %" vector: mostly repeats
        idx = torch.multinomial(a.tree[P:], n, replacement=True, generator=g)
    else:                                        # every leaf evicted: only max_p and the reports change
        idx = torch.randint(0, P, (n,), device="cuda", generator=g)
    _compare(a, b, idx.contiguous(), loss[:idx.numel()].contiguous())


def test_plan_rejects_what_it_cannot_take():
    (a,) = _twins(10)[:1]
    idx = torch.zeros(CAP + 1, dtype=torch.int64, device="cuda")
    loss = torch.ones(CAP + 1, device="cuda")
    plan = torch.empty(_lib.K2B_PLAN_BYTES, dtype=torch.uint8, device="cuda")
    assert a.lib.a0_pt_update_plan(a.h, idx.data_ptr(), CAP + 1, plan.data_ptr(), _lib.stream_ptr()) == EINVAL
    assert a.lib.a0_pt_update_apply(a.h, idx.data_ptr(), loss.data_ptr(), CAP + 1, ALPHA, EPS, plan.data_ptr(), None, None,
                                    _lib.stream_ptr()) == EINVAL


def _loop(rp, algo, Bn, k, planned, o):
    from agent0_b200.hotloop import ReplayTargetLoop
    lp = ReplayTargetLoop(rp, algo, Bn, k, 4, o, n_step=3, rng_seed=5)
    assert lp._use_plan_default == (Bn * k <= CAP)
    lp._use_plan = planned and lp._use_plan_default
    return lp


@pytest.mark.parametrize("algo,Bn,k", [("c51", 32, 20), ("qr", 32, 20), ("c51", 64, 16), ("c51", 41, 25)])
def test_captured_loop_planned_equals_chunk_schedule(algo, Bn, k):
    """Five consecutive replays (each tree feeds the next draw): draws, IS weights, losses, gradients, tree and max_p are
    identical with the planned write-back and with a0_pt_update_overlapped; the same with report slots.  64 x 16 is the
    largest planned count, 41 x 25 = 1025 indices one more (the chunk schedule on both sides)."""
    T = Bn * k
    o = _outputs(algo, T)
    rp_a, rp_b = _shard(algo), _shard(algo)
    la, lb = _loop(rp_a, algo, Bn, k, False, o), _loop(rp_b, algo, Bn, k, True, o)

    def same():
        torch.cuda.synchronize()
        for f in ("idx", "w", "loss", "grad"):
            assert torch.equal(getattr(la, f), getattr(lb, f)), f
        assert torch.equal(rp_a.tree.view(torch.int32), rp_b.tree.view(torch.int32))
        assert float(rp_a.max_p_tensor) == float(rp_b.max_p_tensor)

    la.capture(warm=1); lb.capture(warm=1)
    same()
    for _ in range(5):
        la.run(); lb.run()
        same()
    ra, rb = la.bind_report(2), lb.bind_report(2)
    la.capture_reporting(warm=1); lb.capture_reporting(warm=1)
    for s in range(5):
        la.run(slot=s % 2); lb.run(slot=s % 2)
        same()
        assert torch.equal(ra[s % 2][0], rb[s % 2][0]) and torch.equal(ra[s % 2][1], rb[s % 2][1])
        assert torch.equal(rb[s % 2][0], lb.idx.cpu()) and torch.equal(rb[s % 2][1], lb.loss.cpu())
