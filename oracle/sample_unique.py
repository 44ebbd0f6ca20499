"""The prioritized draw WITHOUT replacement that a0_pt_sample_unique must match bit for bit.  Test infrastructure only.

The reference draws every batch with torch.multinomial(priority[:top], B, replacement=False)
(agent0/deepq/replay.py:41-43): successive sampling, where each next record is drawn with probability
p_i / (S - sum of the priorities already taken).  That is the same law as i.i.d. draws from p with the
repeats thrown away, so a batch is the first B DISTINCT records of a stream of independent tree
descents.  Later rounds descend the tree with the accepted records masked out: given the accepted set
F, the next distinct record has law p restricted to the complement of F, so the law stays exact.

  * Uniforms.  Candidate j = 0, 1, 2, ... of batch k in sampler call c under `seed` takes words x0, x1 of
    Philox4x32-10(counter {j, 0x80000000 | k, c_lo, c_hi}, key {seed_lo, seed_hi}) and
    u_j = ((x0 >> 5) * 2^26 + (x1 >> 6)) * 2^-53 (float64).  Bit 31 of the second counter word keeps this
    stream disjoint from a0_pt_sample_rng's.
  * Masked descent.  F sorted by position, Pre = its float64 prefix sums in ascending position order
    (sequential).  Node v covers leaves [lo_v, hi_v); its masked mass is
    m(v) = max(0, (double)tree[v] - (Pre[hi_v] - Pre[lo_v])), with Pre indexed by the number of F
    positions below the bound.  t = u_j * m(1); at node v go left iff t < m(2v) || !(m(2v+1) > 0), else
    t -= m(2v) and go right.  Leaf i = v - P.  The candidate is VOID if i is in F or p_i <= 0 (only fp32
    rounding of the inner nodes leads there).  With F empty, m(v) is the tree value itself.
  * Rounds.  Round r draws need = B - |F| candidates, all descending against F as it stood at the start of
    the round; walking them in j order, every non-void candidate not yet accepted is accepted.  The batch
    is F in acceptance order (draw order, as torch.multinomial returns it).
  * Shortfall.  m(1) <= 0 at the start of a round, or 8 consecutive rounds that accept nothing: fewer than
    B records have positive priority.  The remaining rows repeat F[0] (position 0 if nothing was drawn).
  * IS weights (trainer.py:91-94) over the B rows: w = (top * (p / (root + sum_offset)))^-beta in fp32,
    divided by the batch maximum + 1e-8; uniform writes w = 1.
"""
import numpy as np

from .sumtree import philox4x32_10

f32 = np.float32
MAX_IDLE_ROUNDS = 8


def unique_uniforms(seed, call, k, j):
    """u_j of candidate j (array) of batch k (array, broadcast) in sampler call ``call`` under ``seed``: float64."""
    j = np.asarray(j, dtype=np.uint64)
    k = np.broadcast_to(np.asarray(k, dtype=np.uint64), j.shape)
    n = j.size
    ctr = np.stack([j.reshape(-1), (k.reshape(-1) | np.uint64(0x80000000)),
                    np.full(n, call & 0xFFFFFFFF, np.uint64), np.full(n, (call >> 32) & 0xFFFFFFFF, np.uint64)],
                   axis=-1).astype(np.uint32)
    key = np.broadcast_to(np.array([seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF], dtype=np.uint32), (n, 2))
    x = philox4x32_10(ctr, key)
    hi = (x[:, 0] >> np.uint32(5)).astype(np.uint64)
    lo = (x[:, 1] >> np.uint32(6)).astype(np.uint64)
    return (((hi << np.uint64(26)) | lo).astype(np.float64) * 2.0 ** -53).reshape(j.shape)


def _lower_bound(Fs, row, a, b, x):
    """First index in [a, b) of row ``row`` of the sorted matrix Fs whose value is >= x (vectorised)."""
    lo, hi = a.copy(), b.copy()
    while True:
        act = lo < hi
        if not act.any():
            return lo
        mid = (lo + hi) // 2
        go = act & (Fs[row, np.minimum(mid, Fs.shape[1] - 1)] < x)
        lo = np.where(go, mid + 1, lo)
        hi = np.where(act & ~go, mid, hi)


def masked_descend(nodes, P, t, Fs, pre, nF, row):
    """Masked descents of targets t (float64) against the sorted accepted sets Fs[row, :nF[row]] with prefix sums
    pre[row]: returns (leaf positions, in_F).  in_F: the leaf is one of the accepted records."""
    D = int(P).bit_length() - 1
    v = np.ones(t.shape, dtype=np.int64)
    a = np.zeros(t.shape, dtype=np.int64)
    b = nF[row].astype(np.int64)
    t = t.copy()
    for d in range(D):
        mid = ((2 * v + 1) << (D - d - 1)) - P
        s = _lower_bound(Fs, row, a, b, mid)
        L = nodes[2 * v].astype(np.float64)
        R = nodes[2 * v + 1].astype(np.float64)
        mL = np.maximum(0.0, L - (pre[row, s] - pre[row, a]))
        mR = np.maximum(0.0, R - (pre[row, b] - pre[row, s]))
        left = (t < mL) | ~(mR > 0)
        t = np.where(left, t, t - mL)
        v = np.where(left, 2 * v, 2 * v + 1)
        a, b = np.where(left, a, s), np.where(left, s, b)
    return v - P, (b - a) == 1


def sample_unique(nodes, P, seed, call, k_batches, batch, top=None, beta=0.4, sum_offset=0.0, uniform=False):
    """The draw of a0_pt_sample_unique on the tree ``nodes`` (f32 [2P], node 1 = root, leaf j at P + j).
    Returns (idx i64[K*B], prio f32[K*B], weights f32[K*B], stats i32[K, 2] = {rounds, candidates}, shortfall bool[K])."""
    nodes = np.asarray(nodes, dtype=f32)
    K, B = int(k_batches), int(batch)
    root = nodes[1]
    F = [[] for _ in range(K)]                         # acceptance order
    Fset = [set() for _ in range(K)]
    j0 = np.zeros(K, dtype=np.int64)
    rounds = np.zeros(K, dtype=np.int32)
    idle = np.zeros(K, dtype=np.int64)
    short = np.zeros(K, dtype=bool)
    Fs = np.full((K, B), P, dtype=np.int64)            # sorted accepted positions, padded with P
    pre = np.zeros((K, B + 1), dtype=np.float64)
    nF = np.zeros(K, dtype=np.int64)
    active = list(range(K))
    while active:
        m1 = np.maximum(0.0, np.float64(root) - pre[active, nF[active]])
        keep = []
        for q, k in enumerate(active):
            if m1[q] > 0:
                keep.append(k)
            else:
                short[k] = True
        active = keep
        if not active:
            break
        act = np.array(active, dtype=np.int64)
        need = B - nF[act]
        row = np.repeat(act, need)
        off = np.arange(row.size) - np.repeat(np.cumsum(need) - need, need)
        j = j0[row] + off
        u = unique_uniforms(seed, call, row, j)
        m1 = np.maximum(0.0, np.float64(root) - pre[row, nF[row]])
        leaf, in_f = masked_descend(nodes, P, u * m1, Fs, pre, nF, row)
        void = in_f | ~(nodes[P + leaf] > 0)
        keep = []
        c = 0
        for q, k in enumerate(active):
            acc = 0
            for i in range(int(need[q])):
                if not void[c + i] and int(leaf[c + i]) not in Fset[k]:
                    F[k].append(int(leaf[c + i]))
                    Fset[k].add(int(leaf[c + i]))
                    acc += 1
            c += int(need[q])
            rounds[k] += 1
            j0[k] += need[q]
            idle[k] = 0 if acc else idle[k] + 1
            if len(F[k]) == B:
                continue
            if idle[k] == MAX_IDLE_ROUNDS:
                short[k] = True
                continue
            srt = np.sort(np.array(F[k], dtype=np.int64))
            n = srt.size
            Fs[k, :n] = srt
            pre[k, 0] = 0.0
            pre[k, 1:n + 1] = np.add.accumulate(nodes[P + srt].astype(np.float64))
            nF[k] = n
            keep.append(k)
        active = keep
    idx = np.empty((K, B), dtype=np.int64)
    for k in range(K):
        fill = F[k][0] if F[k] else 0
        idx[k] = F[k] + [fill] * (B - len(F[k]))
    prio = nodes[P + idx]
    if uniform:
        w = np.ones((K, B), dtype=f32)
    else:
        top = f32(top)
        denom = f32(root + f32(sum_offset))
        w = np.power(top * (prio / denom), f32(-beta)).astype(f32)
        w = (w / (w.max(axis=1, keepdims=True) + f32(1e-8))).astype(f32)
    stats = np.stack([rounds, j0.astype(np.int32)], axis=1).astype(np.int32)
    return idx.reshape(-1), prio.reshape(-1), w.reshape(-1), stats, short


def successive_probability(p, seq):
    """P(the ordered tuple seq) under successive sampling without replacement from weights p."""
    p = np.asarray(p, dtype=np.float64)
    S, out = p.sum(), 1.0
    for i in seq:
        out *= p[i] / S
        S -= p[i]
    return out
