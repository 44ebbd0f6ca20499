"""numpy fp32 restatement of the six train_step target/loss rules.  Test infrastructure only.

Each function takes the *network outputs* the reference's train_step consumes and returns
(per-sample loss, d[(loss*w).sum()]/d[online output]) -- the closed-form gradients reproduce
torch.autograd on the reference graph (BaseLearner.train, agent0/deepq/agent.py:152-155:
the loss is SUM-reduced with the IS weights).  Pinned against tests/golden/loss_*.npz and
static_fns.npz, which come from the unmodified reference.

Conventions: f32 everywhere; G = float32(discount**n_step) (a python double scalar times an
fp32 tensor is evaluated in fp32 by torch); m = 1 - terminal.
"""
import numpy as np

f32 = np.float32


def _G(discount, n_step):
    return f32(discount ** n_step)


def huber(x):
    """F.smooth_l1_loss(beta=1), elementwise."""
    ax = np.abs(x)
    return np.where(ax < 1, f32(0.5) * x * x, ax - f32(0.5)).astype(f32)


def softmax(x, axis=-1):
    z = x - x.max(axis=axis, keepdims=True)
    e = np.exp(z).astype(f32)
    return (e / e.sum(axis=axis, keepdims=True, dtype=f32)).astype(f32)


def log_softmax(x, axis=-1):
    z = x - x.max(axis=axis, keepdims=True)
    return (z - np.log(np.exp(z).sum(axis=axis, keepdims=True, dtype=f32))).astype(f32)


def log_softmax_stable(logits, tau=0.01):
    """agent.py:116-119: (l-max) - tau*logsumexp((l-max)/tau)."""
    z = (logits - logits.max(axis=-1, keepdims=True)).astype(f32)
    s = (z / f32(tau)).astype(f32)
    smax = s.max(axis=-1, keepdims=True)
    lse = smax + np.log(np.exp(s - smax).sum(axis=-1, keepdims=True, dtype=f32))
    return (z - f32(tau) * lse).astype(f32)


def huber_qr_loss(q, q_target, taus):
    """agent.py:110-114 with q [B,1,Nj], q_target [B,Ni,1], taus broadcastable to [B,1,Nj]."""
    u = (q - q_target).astype(f32)                       # [B,Ni,Nj] = q_j - T_i
    rho = huber(u) * np.abs(taus - (q_target < q).astype(f32))
    return rho.sum(-1, dtype=f32).mean(-1, dtype=f32).reshape(-1).astype(f32)


def _huber_qr_grad(qj, Ti, tauj, w):
    """d[(L*w).sum()]/dq_j, q_j [B,Nj], T_i [B,Ni], tau_j [B,Nj] -> [B,Nj]."""
    u = qj[:, None, :] - Ti[:, :, None]
    k = np.abs(tauj[:, None, :] - (u > 0).astype(f32)) * np.clip(u, -1, 1)
    return (w[:, None] / f32(Ti.shape[1]) * k.sum(1, dtype=f32)).astype(f32)


def _td_target(r, d, G, boot):
    return (r + (G * (f32(1) - d)) * boot).astype(f32)


def dqn(q, qt_next, qsel, a, r, d, w, discount, n_step):
    """agent.py:173-190.  qsel = model.qval(next_obs) for double_q, else None (use qt_next)."""
    B = q.shape[0]; bi = np.arange(B)
    a_star = np.argmax(qt_next if qsel is None else qsel, axis=-1)
    T = _td_target(r, d, _G(discount, n_step), qt_next[bi, a_star])
    x = (q[bi, a] - T).astype(f32)
    grad = np.zeros_like(q)
    grad[bi, a] = w * np.clip(x, -1, 1)
    return huber(x), grad


def mdqn(q, qt_next, qt_cur, a, r, d, w, discount, n_step, tau, lo):
    """agent.py:194-215 (softmax at temperature 1, bonus scaled by tau: SURVEY Q11)."""
    B = q.shape[0]; bi = np.arange(B)
    ent = (qt_next - log_softmax_stable(qt_next, tau)).astype(f32)
    v_next = (softmax(qt_next) * ent).sum(-1, dtype=f32)
    add_on = np.clip(log_softmax_stable(qt_cur, tau)[bi, a], f32(lo), f32(0))
    T = ((r + f32(tau) * add_on) + (_G(discount, n_step) * (f32(1) - d)) * v_next).astype(f32)
    x = (q[bi, a] - T).astype(f32)
    grad = np.zeros_like(q)
    grad[bi, a] = w * np.clip(x, -1, 1)
    return huber(x), grad


def c51_project(p_next, r, d, atoms, vmin, vmax, G):
    """agent.py:230-264: categorical projection of r + G*m*z onto the support. Returns m [B,M]."""
    B, M = p_next.shape
    delta = f32((vmax - vmin) / (M - 1))
    tz = np.clip(r[:, None] + (G * (f32(1) - d))[:, None] * atoms[None, :], f32(vmin), f32(vmax)).astype(f32)
    base = ((tz - f32(vmin)) / delta).astype(f32)
    lo = np.floor(base).astype(np.int64); up = np.ceil(base).astype(np.int64)
    lo[(up > 0) & (lo == up)] -= 1
    up[(lo < (M - 1)) & (lo == up)] += 1
    m = np.zeros((B, M), dtype=f32)
    for b in range(B):       # index_add_ order: all lo terms, then all up terms
        np.add.at(m[b], lo[b], (p_next[b] * (up[b].astype(f32) - base[b])).astype(f32))
        # delta is rounded to fp32, so an atom clamped at vmax can get a base just above M-1 and up == M: that
        # upper term is dropped (DESIGN section 5)
        keep = up[b] < M
        np.add.at(m[b], up[b][keep], (p_next[b] * (base[b] - lo[b].astype(f32))).astype(f32)[keep])
    return m


def c51(logits, tgt_logits, qsel, a, r, d, w, discount, n_step, atoms, vmin, vmax):
    """agent.py:219-269.  logits/tgt_logits [B,A,M]; returns loss, grad [B,A,M], target_prob."""
    B = logits.shape[0]; bi = np.arange(B)
    prob_next = softmax(tgt_logits)
    a_star = np.argmax(qsel, -1) if qsel is not None else \
        np.argmax((prob_next * atoms[None, None, :]).sum(-1, dtype=f32), -1)
    m = c51_project(prob_next[bi, a_star], r, d, atoms, vmin, vmax, _G(discount, n_step))
    logp = log_softmax(logits[bi, a])
    loss = -(m * logp).sum(-1, dtype=f32)
    grad = np.zeros_like(logits)
    grad[bi, a] = w[:, None] * (np.exp(logp) * m.sum(-1, keepdims=True, dtype=f32) - m)
    return loss.astype(f32), grad, m


def qr(q, qt_next, qsel, a, r, d, w, discount, n_step):
    """agent.py:273-293.  q/qt_next [B,A,N], tau_j=(2j+1)/2N (model.py:185-188)."""
    B, _, N = q.shape; bi = np.arange(B)
    a_star = np.argmax(qsel, -1) if qsel is not None else np.argmax(qt_next.mean(-1, dtype=f32), -1)
    T = _td_target(r[:, None], d[:, None], _G(discount, n_step), qt_next[bi, a_star])
    tau = ((2 * np.arange(N) + 1).astype(f32) / f32(2.0 * N)).astype(f32)
    qa = q[bi, a]
    loss = huber_qr_loss(qa[:, None, :], T[:, :, None], tau[None, None, :])
    grad = np.zeros_like(q)
    grad[bi, a] = _huber_qr_grad(qa, T, np.broadcast_to(tau, qa.shape), w)
    return loss, grad


def iqn(q_cur, taus_cur, q_next, qsel, a, r, d, w, discount, n_step):
    """agent.py:297-327.  q_cur [B,N,A], taus_cur [B,N], q_next [B,N',A], qsel [B,A]."""
    B = q_cur.shape[0]; bi = np.arange(B)
    a_star = np.argmax(qsel, -1)
    T = _td_target(r[:, None], d[:, None], _G(discount, n_step), q_next[bi, :, a_star])
    qa = q_cur[bi, :, a]
    loss = huber_qr_loss(qa[:, None, :], T[:, :, None], taus_cur[:, None, :])
    grad = np.zeros_like(q_cur)
    grad[bi, :, a] = _huber_qr_grad(qa, T, taus_cur, w)
    return loss, grad


def fqf(q_hat, taus, taus_hat, q_next, q_bar, qsel, a, r, d, w, discount, n_step):
    """agent.py:340-388.  q_hat/q_next [B,F,A] at taus_hat [B,F]; q_bar [B,F-1,A] at the
    interior taus[:,1:-1]; taus [B,F+1].  Returns q loss, grad wrt q_hat, fraction loss,
    d[(fraction_loss*w).sum()]/d taus [B,F+1]."""
    loss, grad = iqn(q_hat, taus_hat, q_next, qsel, a, r, d, w, discount, n_step)
    B = q_hat.shape[0]; bi = np.arange(B)
    qh = q_hat[bi, :, a]; qb = q_bar[bi, :, a]
    v1 = qb - qh[:, :-1]
    s1 = qb > np.concatenate((qh[:, :1], qb[:, :-1]), 1)
    v2 = qb - qh[:, 1:]
    s2 = qb < np.concatenate((qb[:, 1:], qh[:, -1:]), 1)
    g = (np.where(s1, v1, -v1) + np.where(s2, v2, -v2)).astype(f32)
    frac = (g * taus[:, 1:-1]).sum(1, dtype=f32)
    gt = np.zeros_like(taus)
    gt[:, 1:-1] = w[:, None] * g
    return loss, grad, frac.astype(f32), gt


def huber_qr_sorted(qj, Ti, tauj, w):
    """The quantile-Huber pair sums of agent.py:110-114 in O(N log N) per sample: SPECIFICATION of the planned
    sorted-target K4 (DESIGN section 11), checked on the CPU against the pairwise form above.

    qj [B,Nj] online quantiles, Ti [B,Ni] targets, tauj [B,Nj] (or [Nj]), w [B] IS weights.  Returns
    (loss [B], grad [B,Nj]) = (huber_qr_loss, _huber_qr_grad).  For a fixed q the sorted targets split
    into four ranges of u = q - T:  u >= 1 (linear, weight 1-tau), 0 < u < 1 (quadratic, 1-tau),
    -1 < u <= 0 (quadratic, tau), u <= -1 (linear, tau); over each range the Huber terms are polynomials
    in q whose coefficients are prefix sums of T and T^2.  The prefix sums are float64 and centred on the
    sorted target c at position Ni//2 (sums of T-c and (T-c)^2, polynomial in q-c; both differences are exact
    for fp32 inputs): the quadratic ranges subtract numbers of size N*(T-c)^2 to obtain terms of size
    (q-T)^2, where uncentred sums of size N*T^2 lose the 1e-5 contract from |T| ~ 1e5.  The ranges are
    found on the uncentred values."""
    qj = np.asarray(qj, dtype=np.float64)
    B, Nj = qj.shape
    Ni = Ti.shape[1]
    tau = np.broadcast_to(np.asarray(tauj, dtype=np.float64), (B, Nj))
    loss = np.zeros(B, dtype=np.float64)
    grad = np.zeros((B, Nj), dtype=np.float64)
    for b in range(B):
        T = np.sort(np.asarray(Ti[b], dtype=np.float64))
        c = T[Ni // 2]
        S1 = np.concatenate(([0.0], np.cumsum(T - c)))
        S2 = np.concatenate(([0.0], np.cumsum((T - c) * (T - c))))
        ia = np.searchsorted(T, qj[b] - 1.0, side="right")    # T <= q-1          : u >= 1
        ib = np.searchsorted(T, qj[b], side="left")           # q-1 < T < q       : 0 < u < 1
        ic = np.searchsorted(T, qj[b] + 1.0, side="left")     # q <= T < q+1      : -1 < u <= 0
        q = qj[b] - c
        nA, nB, nC, nD = ia, ib - ia, ic - ib, Ni - ic
        s1B, s2B = S1[ib] - S1[ia], S2[ib] - S2[ia]
        s1C, s2C = S1[ic] - S1[ib], S2[ic] - S2[ib]
        s1D = S1[Ni] - S1[ic]
        A_ = nA * (q - 0.5) - S1[ia]
        B_ = 0.5 * (nB * q * q - 2.0 * q * s1B + s2B)
        C_ = 0.5 * (nC * q * q - 2.0 * q * s1C + s2C)
        D_ = s1D - nD * (q + 0.5)
        loss[b] = ((1.0 - tau[b]) * (A_ + B_) + tau[b] * (C_ + D_)).sum() / Ni
        grad[b] = ((1.0 - tau[b]) * (nA + nB * q - s1B) + tau[b] * (nC * q - s1C - nD)) * (float(w[b]) / Ni)
    return loss.astype(f32), grad.astype(f32)
