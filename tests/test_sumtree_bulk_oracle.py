"""The bulk forms of oracle/sumtree.py (SumTree.build, .update, .sample), which let the GPU tests check trees of up to
2^24 leaves, against the scalar definition they replace there (SumTree.set, .sample_stratified and the write-back
rules spelled out one entry at a time): identical nodes, indices and priorities at every depth from 1 to 16, on
zero runs, magnitudes from 2^-20 to 2^20, exact ties and the extreme uniforms 0 and 1 - 2^-24.  CPU only."""
import numpy as np
import pytest

from oracle.sumtree import SumTree, new_priority

f32 = np.float32
U_MAX = f32(1.0 - 2.0 ** -24)


def _leaves(kind, D, rng):
    """N = P - P/8 leaves (N = P for "ties"), float32."""
    P = 1 << D
    N = P if kind == "ties" else max(2, P - P // 8)
    if kind == "spread":
        v = np.sqrt(np.abs(rng.randn(N)) + 0.01)
        v[rng.rand(N) < 0.03] = 0.0
    elif kind == "holes":                          # aligned zero runs of 32, 1024 and 2^(D-10) leaves, and the left half
        v = np.sqrt(np.abs(rng.randn(N)) + 0.01)
        for unit in (32, 1024, 1 << max(D - 10, 0)):
            for lo in range(0, N, unit):
                if rng.rand() < 0.25:
                    v[lo:lo + unit] = 0.0
        v[:P // 2] = 0.0
        v[N - 1] = 1.0
    elif kind == "range":                          # parents absorb small children, t - L rounds
        v = np.exp2(rng.uniform(-20, 20, N))
    elif kind == "ties":
        v = np.ones(N)
    else:                                          # "single": one live leaf
        v = np.zeros(N)
        v[rng.randint(N)] = 1.5
    return v.astype(f32)


KINDS = ["spread", "holes", "range", "ties", "single"]


@pytest.mark.parametrize("D", range(1, 17))
@pytest.mark.parametrize("kind", KINDS)
def test_bulk_build_and_descent_equal_the_scalar_definition(D, kind):
    rng = np.random.RandomState(100 * D + KINDS.index(kind))
    v = _leaves(kind, D, rng)
    a, b = SumTree(v.size), SumTree(v.size)
    assert a.P == 1 << D
    a.set(np.arange(v.size), v)
    b.build(v)
    assert np.array_equal(a.nodes.view(np.int32), b.nodes.view(np.int32))
    for B, K in ((1, 1), (7, 3), (32, 2), (512, 1)):
        for u in (rng.rand(B * K).astype(f32), np.zeros(B * K, f32), np.full(B * K, U_MAX)):
            idx, prio = b.sample(u, B)
            want = [a.sample_stratified(u[k * B:(k + 1) * B]) for k in range(K)]
            assert np.array_equal(idx, np.concatenate([w[0] for w in want]))
            assert np.array_equal(prio.view(np.int32), np.concatenate([w[1] for w in want]).view(np.int32))
            assert (prio > 0).all()


def _update_scalar(tree, idx, loss, eps, alpha, max_p):
    """The write-back rules one entry at a time, then SumTree.set."""
    last = {}
    for k, p in enumerate(idx):
        if 0 <= p < tree.capacity:
            last[int(p)] = k
            if np.isfinite(loss[k]):
                max_p = max(max_p, f32(loss[k]))
    ids, vals = [], []
    for p, k in last.items():
        if tree.nodes[tree.P + p] > 0 and np.isfinite(loss[k]) and loss[k] >= 0:
            ids.append(p)
            vals.append(new_priority(loss[k:k + 1], eps, alpha)[0])
    if ids:
        tree.set(ids, vals)
    return f32(max_p)


@pytest.mark.parametrize("D", [1, 2, 5, 12, 16])
@pytest.mark.parametrize("alpha", [0.5, 0.6])
def test_bulk_update_equals_the_scalar_rules(D, alpha):
    rng = np.random.RandomState(D)
    v = _leaves("spread", D, rng)
    a, b = SumTree(v.size), SumTree(v.size)
    a.build(v)
    b.build(v)
    max_a = max_b = f32(0.75)
    P = a.P
    for count in (1, 7, 640, 1025):
        idx = rng.randint(-2, P + 2, count).astype(np.int64)
        loss = (rng.rand(count) * 3).astype(f32)
        if count > 8:
            idx[-4:] = idx[0]                                   # duplicates: the last one wins
            loss[-1] = np.nan                                   # ... and its NaN leaves the old leaf
            loss[2], loss[3], loss[4] = np.inf, 50.0, -0.5      # inf beside the largest finite loss
            idx[3] = rng.randint(0, v.size)
            idx[5:7] = (idx[5] & ~1) + np.array([0, 1])         # siblings
        max_a = _update_scalar(a, idx, loss, 0.01, alpha, max_a)
        max_b = b.update(idx, loss, 0.01, alpha, max_b)
        assert np.array_equal(a.nodes.view(np.int32), b.nodes.view(np.int32)), count
        assert max_a == max_b
        if count > 8:
            assert max_b == f32(50.0)


def test_nan_winner_keeps_the_old_leaf_and_evicted_leaves_stay_zero():
    t = SumTree(8)
    t.build(np.array([1, 2, 0, 4, 5, 6, 7, 8], f32))
    mp = t.update([1, 1, 2, 9, -1], np.array([3.0, np.nan, 1.0, 7.0, 7.0], f32), 0.01, 0.5, 1.0)
    assert t.leaves()[1] == 2.0 and t.leaves()[2] == 0.0 and mp == 3.0
    assert t.root == f32(33.0)
