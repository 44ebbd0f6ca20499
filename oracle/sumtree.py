"""The fp32 sum-tree the CUDA sampler (K2a/K2b) must match bit-for-bit.  Test infrastructure only.

No reference counterpart: the reference keeps a flat fp32 priority vector and its intended
law is P(i) = priority[i] / sum(priority) via torch.multinomial without replacement
(agent0/deepq/replay.py:39-43, dead code behind a RandomSampler).  The tree is the B200
design's replacement; its arithmetic is *defined* here so that sampled indices are
reproducible:

  * implicit complete binary tree over P = next_pow2(capacity) leaves, node 1 = root,
    children of i are 2i and 2i+1, leaf j lives at P + j;
  * every internal node is fl32(left + right), recomputed from its children (never a delta);
  * stratified draw b of B with uniform u_b:  t = fl32(fl32(fl32(b + u_b) / B) * root);
    descent: go left iff (t < left) or (right <= 0); when going right, t = fl32(t - left).
"""
import numpy as np

f32 = np.float32


def next_pow2(n):
    p = 1
    while p < n:
        p *= 2
    return p


class SumTree:
    def __init__(self, capacity):
        self.capacity = capacity
        self.P = next_pow2(max(capacity, 2))
        self.nodes = np.zeros(2 * self.P, dtype=f32)

    @property
    def root(self):
        return self.nodes[1]

    def leaves(self):
        return self.nodes[self.P:self.P + self.capacity]

    def set(self, idx, values):
        """Set leaves (sequential: the last occurrence of a duplicated index wins), then
        recompute every ancestor from its children, level by level."""
        idx = np.asarray(idx, dtype=np.int64)
        values = np.asarray(values, dtype=f32)
        for i, v in zip(idx, values):
            self.nodes[self.P + i] = v
        level = np.unique((self.P + idx) >> 1)
        while True:
            self.nodes[level] = self.nodes[2 * level] + self.nodes[2 * level + 1]
            if level[0] == 1:
                break
            level = np.unique(level >> 1)

    def descend(self, t):
        node = 1
        t = f32(t)
        while node < self.P:
            left, right = self.nodes[2 * node], self.nodes[2 * node + 1]
            if t < left or right <= 0:
                node = 2 * node
            else:
                t = f32(t - left)
                node = 2 * node + 1
        return node - self.P

    def sample_stratified(self, u):
        u = np.asarray(u, dtype=f32)
        B = u.shape[0]
        root = self.root
        idx = np.empty(B, dtype=np.int64)
        for b in range(B):
            t = f32(f32(f32(b) + u[b]) / f32(B)) * root
            idx[b] = self.descend(f32(t))
        return idx, self.nodes[self.P + idx].copy()

    # ---- bulk forms: the same float32 operations as set / sample_stratified, one numpy operation per tree level,
    #      so that trees of up to 2^24 leaves can be built and descended in well under a second
    def build(self, leaves):
        """set(arange(len(leaves)), leaves) on an empty tree: every node recomputed, level by level."""
        leaves = np.asarray(leaves, dtype=f32)
        self.nodes[:] = 0
        self.nodes[self.P:self.P + leaves.size] = leaves
        n = self.P // 2
        while n >= 1:
            self.nodes[n:2 * n] = self.nodes[2 * n:4 * n:2] + self.nodes[2 * n + 1:4 * n:2]
            n //= 2

    def _recompute(self, leaf_pos):
        level = np.unique((self.P + np.asarray(leaf_pos, dtype=np.int64)) >> 1)
        while level.size:
            self.nodes[level] = self.nodes[2 * level] + self.nodes[2 * level + 1]
            level = np.unique(level[level > 1] >> 1)

    def update(self, idx, loss, eps, alpha, max_p):
        """The priority write-back (a0_pt_update and every K2b schedule); returns the new max_p.
          * positions outside [0, capacity) are ignored;
          * of several entries for one position the last one wins;
          * a winner whose loss is NaN, infinite or negative leaves the old leaf (no fall-back to an earlier entry);
          * a leaf that is 0 (evicted since it was sampled) stays 0;
          * max_p = max(max_p, every finite loss at a position in range) (replay.py:59)."""
        idx = np.asarray(idx, dtype=np.int64)
        loss = np.asarray(loss, dtype=f32)
        ok = (idx >= 0) & (idx < self.capacity)
        finite = ok & np.isfinite(loss)
        if finite.any():
            max_p = max(f32(max_p), f32(loss[finite].max()))
        pos, k = idx[ok], np.flatnonzero(ok)
        if pos.size == 0:
            return f32(max_p)
        rev_first = np.unique(pos[::-1], return_index=True)[1]
        win = k[pos.size - 1 - rev_first]                        # the last entry of every distinct position
        p, x = idx[win], loss[win]
        good = (x >= 0) & np.isfinite(x) & (self.nodes[self.P + p] > 0)
        self.nodes[self.P + p[good]] = new_priority(x[good], eps, alpha)
        self._recompute(p)
        return f32(max_p)

    def sample(self, u, batch):
        """sample_stratified over consecutive batches of ``batch`` uniforms (draw g is stratum g % batch),
        all draws descending together: t = fl32(fl32(fl32(b + u) / B) * root); go left iff t < L or not (R > 0);
        going right, t = fl32(t - L)."""
        u = np.asarray(u, dtype=f32)
        b = (np.arange(u.size) % batch).astype(f32)
        t = ((b + u) / f32(batch)) * self.root
        node = np.ones(u.size, dtype=np.int64)
        for _ in range(self.P.bit_length() - 1):
            L, R = self.nodes[2 * node], self.nodes[2 * node + 1]
            right = ~((t < L) | ~(R > 0))
            t = np.where(right, t - L, t).astype(f32)
            node = 2 * node + right
        idx = node - self.P
        return idx, self.nodes[node].copy()


def new_priority(loss, eps, alpha):
    """replay.py:56-58: (loss+eps)^alpha; sqrt when alpha == 0.5 as torch's CPU pow does."""
    x = np.asarray(loss, dtype=f32) + f32(eps)
    return np.sqrt(x) if alpha == 0.5 else np.power(x, f32(alpha)).astype(f32)


def philox4x32_10(counter, key):
    """Philox4x32-10 (Salmon, Moraes, Dror, Shaw: "Parallel random numbers: as easy as 1, 2, 3", SC'11;
    the Random123 reference implementation's constants).  counter: uint32 [..., 4], key: uint32
    [..., 2] -> uint32 [..., 4].  The reference repository has no counterpart: this defines the
    uniforms of a0_pt_sample_rng."""
    c = [np.asarray(counter[..., i], dtype=np.uint64) for i in range(4)]
    k = [np.asarray(key[..., i], dtype=np.uint64) for i in range(2)]
    M0, M1, W0, W1, mask = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), np.uint64(0x9E3779B9), np.uint64(0xBB67AE85), \
        np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0, p1 = M0 * c[0], M1 * c[2]
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & mask, p1 >> np.uint64(32), p1 & mask
        c = [hi1 ^ c[1] ^ k[0], lo1, hi0 ^ c[3] ^ k[1], lo0]
        k = [(k[0] + W0) & mask, (k[1] + W1) & mask]
    return np.stack([x.astype(np.uint32) for x in c], axis=-1)


def philox_uniform(seed, call, n):
    """The n uniforms of sampler call number ``call`` under ``seed`` (a0_pt_sample_rng): draw g is
    (philox(counter {g, 0, call_lo, call_hi}, key {seed_lo, seed_hi})[0] >> 8) * 2^-24, float32."""
    g = np.arange(n, dtype=np.uint64)
    ctr = np.stack([g & np.uint64(0xFFFFFFFF), np.zeros(n, np.uint64), np.full(n, call & 0xFFFFFFFF, np.uint64),
                    np.full(n, (call >> 32) & 0xFFFFFFFF, np.uint64)], axis=-1).astype(np.uint32)
    key = np.broadcast_to(np.array([seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF], dtype=np.uint32), (n, 2))
    x = philox4x32_10(ctr, key)[..., 0]
    return ((x >> np.uint32(8)).astype(np.float32) * np.float32(2.0 ** -24)).astype(np.float32)
