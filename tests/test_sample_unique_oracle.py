"""The draw without replacement (oracle/sample_unique.py, the definition a0_pt_sample_unique matches bit for bit)
follows the law of torch.multinomial(p, B, replacement=False) -- the reference's ReplayDataset.__iter__,
agent0/deepq/replay.py:41-43 -- and its rounds, masking and shortfall behave as specified.  CPU only."""
import itertools
from collections import Counter

import numpy as np
import pytest
import torch
from scipy import stats

from oracle.sample_unique import masked_descend, sample_unique, successive_probability, unique_uniforms
from oracle.sumtree import SumTree

THRESHOLD = 1e-6
BATCHES = 100_000


def _tree(p):
    t = SumTree(len(p))
    t.set(np.arange(len(p)), np.asarray(p, dtype=np.float32))
    return t


def _chi2_pvalue(observed, expected):
    """Pearson chi-square with the cells of expected count < 5 pooled into one."""
    observed, expected = np.asarray(observed, float), np.asarray(expected, float)
    small = expected < 5
    o = np.append(observed[~small], observed[small].sum())
    e = np.append(expected[~small], expected[small].sum())
    if e[-1] == 0:
        o, e = o[:-1], e[:-1]
    chi = float(((o - e) ** 2 / e).sum())
    return stats.chi2.sf(chi, len(e) - 1)


@pytest.mark.parametrize("p,B", [([1.0, 2.0, 3.0, 4.0, 5.0, 6.5], 3),
                                 ([0.5, 1.5, 1.0, 3.25, 2.0, 0.75, 4.0, 1.25], 2),
                                 ([2.0, 1.0, 3.0, 1.5, 2.5, 4.0, 3.5], 4)])
def test_ordered_batches_follow_successive_sampling_and_torch_multinomial(p, B):
    t = _tree(p)
    idx, prio, w, st, short = sample_unique(t.nodes, t.P, seed=20261020 + B, call=3, k_batches=BATCHES, batch=B,
                                            top=len(p), beta=0.4)
    assert not short.any()
    rows = idx.reshape(-1, B)
    assert all(len(set(r)) == B for r in rows[:2000])
    np.testing.assert_array_equal(prio, np.asarray(p, np.float32)[idx])
    tuples = list(itertools.permutations(range(len(p)), B))
    got = Counter(map(tuple, rows))
    assert sum(got.values()) == BATCHES and set(got) <= set(tuples)
    obs = np.array([got.get(s, 0) for s in tuples])
    exp = np.array([BATCHES * successive_probability(p, s) for s in tuples])
    assert abs(exp.sum() - BATCHES) < 1e-6 * BATCHES
    assert _chi2_pvalue(obs, exp) > THRESHOLD
    # two-sample test against torch.multinomial(p, B, replacement=False) on the CPU
    g = torch.Generator().manual_seed(7 + B)
    ref = torch.multinomial(torch.tensor(p, dtype=torch.float64).expand(BATCHES, len(p)), B, replacement=False,
                            generator=g).numpy()
    want = Counter(map(tuple, ref))
    table = np.array([[got.get(s, 0) for s in tuples], [want.get(s, 0) for s in tuples]])
    table = table[:, table.sum(axis=0) > 0]
    assert stats.chi2_contingency(table)[1] > THRESHOLD


def test_uniforms_are_53_bit_and_disjoint_from_the_stratified_stream():
    u = unique_uniforms(5, 2, np.arange(4), np.arange(4))
    assert u.dtype == np.float64 and ((u >= 0) & (u < 1)).all()
    assert (np.ldexp(u, 53) == np.round(np.ldexp(u, 53))).all()
    assert len(set((u * 2.0 ** 24).astype(np.int64) % 7)) > 1            # not 24-bit values scaled up
    # batch index is part of the counter: the same candidate in two batches differs
    assert unique_uniforms(5, 2, 0, [0])[0] != unique_uniforms(5, 2, 1, [0])[0]


def test_masked_descents_never_return_an_accepted_record():
    """With integer priorities every node is exact, so the masked masses are exact and no candidate is void:
    the descents land only on records outside F, with the law p restricted to the complement."""
    rng = np.random.RandomState(3)
    p = rng.randint(1, 50, 300).astype(np.float32)
    t = _tree(p)
    F = np.sort(rng.choice(300, 40, replace=False))
    K = 1
    Fs = np.full((K, 64), t.P, dtype=np.int64)
    Fs[0, :40] = F
    pre = np.zeros((K, 65))
    pre[0, 1:41] = np.add.accumulate(p[F].astype(np.float64))
    n = 200_000
    row = np.zeros(n, dtype=np.int64)
    m1 = float(t.root) - pre[0, 40]
    leaf, in_f = masked_descend(t.nodes, t.P, rng.rand(n) * m1, Fs, pre, np.array([40]), row)
    assert not in_f.any() and not np.isin(leaf, F).any() and (leaf < 300).all()
    rest = np.setdiff1d(np.arange(300), F)
    freq = np.bincount(leaf, minlength=300)[rest]
    exp = n * p[rest] / p[rest].sum()
    assert _chi2_pvalue(freq, exp) > THRESHOLD


def test_rounds_mask_what_was_taken():
    """One leaf holding 99.9 % of the mass: round 1 takes it (and its repeats are discarded), the next rounds draw
    from the rest with it masked out -- at most 3 rounds, never a record twice."""
    N, B, K = 1024, 32, 64
    p = np.ones(N, dtype=np.float32)
    p[517] = 999.0 * (N - 1)
    t = _tree(p)
    idx, prio, w, st, short = sample_unique(t.nodes, t.P, seed=11, call=0, k_batches=K, batch=B, top=N, beta=0.6)
    rows = idx.reshape(K, B)
    assert not short.any()
    assert all(len(set(r)) == B for r in rows)
    assert (rows[:, 0] == 517).mean() > 0.99                           # first draw: the heavy record
    assert st[:, 0].max() <= 3 and (st[:, 0] >= 2).all()
    assert (st[:, 1] >= B).all() and (st[:, 1] < 3 * B).all()
    wk = w.reshape(K, B)
    np.testing.assert_allclose(wk.max(axis=1), 1.0, rtol=1e-6)


def test_shortfall_is_reported_instead_of_looping():
    N, B = 16, 5
    p = np.zeros(N, dtype=np.float32)
    p[[3, 9, 12]] = [1.0, 2.0, 4.0]
    t = _tree(p)
    idx, prio, w, st, short = sample_unique(t.nodes, t.P, seed=1, call=0, k_batches=4, batch=B, top=3, beta=0.4)
    assert short.all()
    rows = idx.reshape(4, B)
    for r in rows:
        assert sorted(r[:3]) == [3, 9, 12] and (r[3:] == r[0]).all()
    assert (prio > 0).all() and (st[:, 0] <= 2).all()
    # exactly B positive records: no shortfall, all of them
    p[[0, 5]] = 0.5
    t = _tree(p)
    idx, _, _, st, short = sample_unique(t.nodes, t.P, seed=1, call=0, k_batches=4, batch=B, top=5, beta=0.4)
    assert not short.any() and all(sorted(r) == [0, 3, 5, 9, 12] for r in idx.reshape(4, B))
    # nothing positive at all: the first round already sees m(1) = 0
    t = _tree(np.zeros(N, dtype=np.float32))
    idx, _, _, st, short = sample_unique(t.nodes, t.P, seed=1, call=0, k_batches=1, batch=B, top=0, beta=0.4)
    assert short.all() and (st[:, 0] == 0).all() and (idx == 0).all()


def test_uniform_shard_draws_a_uniform_subset_with_unit_weights():
    N, B, K = 10, 3, 30_000
    t = _tree(np.ones(N, dtype=np.float32))
    idx, _, w, st, short = sample_unique(t.nodes, t.P, seed=4, call=9, k_batches=K, batch=B, uniform=True)
    assert (w == 1).all() and not short.any()
    subsets = Counter(tuple(sorted(r)) for r in idx.reshape(K, B))
    assert len(subsets) == 120
    assert _chi2_pvalue([subsets[s] for s in sorted(subsets)], [K / 120] * 120) > THRESHOLD


def test_argument_errors_of_the_entry_point_do_not_need_a_gpu():
    from agent0_b200 import _lib
    lib = _lib.load()
    f = lib.a0_pt_sample_unique
    assert f(None, 1, -1, 4, 2, 1.0, 0.4, 0.0, 0, None, None, None, None, None) == -1
    assert b"handle is NULL" in lib.a0_last_error()
    assert f(None, 1, -1, 2048, 2048, 1.0, 0.4, 0.0, 0, None, None, None, None, None) == -1
    assert b"batch 2048 outside [1, 1024]" in lib.a0_last_error()
    assert f(None, 1, -1, 10, 4, 1.0, 0.4, 0.0, 0, None, None, None, None, None) == -1
    assert b"must be a multiple of batch" in lib.a0_last_error()
    assert f(None, 1, -1, 4097 * 2, 2, 1.0, 0.4, 0.0, 0, None, None, None, None, None) == -1
    assert b"at most 4096 per call" in lib.a0_last_error()
    assert f(None, 1, -1, 0, 0, 1.0, 0.4, 0.0, 0, None, None, None, None, None) == -1
