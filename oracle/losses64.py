"""float64 evaluation of the six target/loss rules, with an error scale per output element.  Test infrastructure only.

Takes the same fp32 inputs as oracle/losses.py.  The discrete decisions are taken from fp32 values, as the kernels
take them: the selected action a* (first maximum), the C51 bins l and u from the fp32 base (formed with the kernels'
fp32 operations, delta = fl32(fl32(vmax - vmin) / (M - 1)) included), the side of q - T, the FQF comparisons, and the
TD target T = r + (G*(1-d))*boot with each operation rounded (DESIGN section 5).  Everything downstream -- softmax,
log-softmax, projection weights, cross-entropy, Huber pair sums, gradients, fraction loss, (loss + eps)^alpha -- is
float64.

Every output is an ``R(v, s, n)``: per element the float64 value v, the sum s of the absolute values of the terms
the value accumulates (operands of a difference count with their own magnitude), and their number n.  An fp32
evaluation of the same rule, in any summation order, lies within a small multiple of n * 2^-24 * s of v; an element
with s = 0 is exactly 0.  The functions take the bootstrap factor G = gamma^n as the fp32 scalar the C ABI takes."""
from collections import namedtuple

import numpy as np

from oracle import losses as OL

f32 = np.float32
R = namedtuple("R", "v s n")


def _d(x):
    return np.asarray(x, dtype=np.float64)


def _td_huber(q, a, w, T, sT, nT):
    """huber(q[a] - T) and w * clamp(q[a] - T) with T float64 of error scale sT."""
    B, A = q.shape
    bi = np.arange(B)
    qa = _d(q[bi, a])
    x = qa - T
    ax = np.abs(x)
    c = np.minimum(ax, 1.0)
    sx = np.abs(qa) + sT
    loss = R(c * (ax - 0.5 * c), c * (ax - 0.5 * c) + c * sx, np.full(B, nT + 4))
    gv = np.zeros((B, A)); gs = np.zeros((B, A))
    gv[bi, a] = _d(w) * np.clip(x, -1.0, 1.0)
    gs[bi, a] = np.abs(_d(w)) * (sx + 1.0)
    return {"loss": loss, "grad": R(gv, gs, np.full((B, A), nT + 4))}


def dqn(q, qt_next, qsel, a, r, d, w, G):
    """agent.py:173-190; qsel None: select on qt_next."""
    bi = np.arange(q.shape[0])
    a_star = np.argmax(qt_next if qsel is None else qsel, -1)
    T = _d(OL._td_target(r, d, f32(G), qt_next[bi, a_star]))
    return _td_huber(q, a, w, T, np.abs(T), 0)


def _log_softmax_stable(l, tau):
    """agent.py:116-119 in float64 of the fp32 row l: value, error scale, and the softmax at temperature tau."""
    z = _d(l) - _d(l).max(-1, keepdims=True)
    e = np.exp(z / tau)
    lse = np.log(e.sum(-1, keepdims=True))
    pt = e / e.sum(-1, keepdims=True)
    s = np.abs(z) + tau * (np.abs(lse) + 1.0) + (pt * np.abs(z)).sum(-1, keepdims=True)
    return z - tau * lse, s


def mdqn(q, qt_next, qt_cur, a, r, d, w, G, tau, lo):
    """agent.py:194-215 (softmax at temperature 1, bonus scaled by tau: SURVEY Q11)."""
    B, A = q.shape
    bi = np.arange(B)
    tau, lo = float(f32(tau)), float(f32(lo))                 # the fp32 scalars the kernel takes
    tn = _d(qt_next)
    tlp, s_tlp = _log_softmax_stable(qt_next, tau)
    zn = tn - tn.max(-1, keepdims=True)
    p = np.exp(zn) / np.exp(zn).sum(-1, keepdims=True)
    boot = (p * (tn - tlp)).sum(-1)
    s_boot = (p * (np.abs(tn) + s_tlp + np.abs(tn - tlp))).sum(-1)
    tlc, s_tlc = _log_softmax_stable(qt_cur, tau)
    bonus = tau * np.clip(tlc[bi, a], lo, 0.0)
    s_bonus = tau * s_tlc[bi, a]
    gm = _d(f32(G) * (f32(1) - d))
    T = (_d(r) + bonus) + gm * boot
    sT = np.abs(_d(r)) + s_bonus + np.abs(gm) * s_boot + np.abs(_d(r) + bonus) + np.abs(gm * boot)
    return _td_huber(q, a, w, T, sT, A + 12)


def c51_bins(r, d, atoms, vmin, vmax, G):
    """The kernels' fp32 projection arithmetic: base [B,M] (fp32), lower and upper bins.  An upper bin equal to M
    (the base of an atom clamped at vmax rounded above M-1) marks a term that is dropped."""
    M = atoms.shape[0]
    delta = f32(f32(f32(vmax) - f32(vmin)) / f32(M - 1))
    gm = (f32(G) * (f32(1) - d)).astype(f32)
    tz = (r[:, None] + gm[:, None] * atoms[None, :]).astype(f32)
    tz = np.minimum(np.maximum(tz, f32(vmin)), f32(vmax))
    base = ((tz - f32(vmin)).astype(f32) / delta).astype(f32)
    lo = np.floor(base).astype(np.int64)
    up = np.ceil(base).astype(np.int64)
    lo[(up > 0) & (lo == up)] -= 1
    up[(lo < M - 1) & (lo == up)] += 1
    return base, lo, up


def _softmax(l):
    z = _d(l) - _d(l).max(-1, keepdims=True)
    e = np.exp(z)
    return e / e.sum(-1, keepdims=True)


def c51(logits, tgt_logits, qsel, a, r, d, w, G, atoms, vmin, vmax):
    """agent.py:219-269.  Returns loss, grad [B,A,M] and the projected distribution target_prob [B,M]."""
    B, A, M = logits.shape
    bi = np.arange(B)
    if qsel is not None:
        a_star = np.argmax(qsel, -1)
    else:
        a_star = np.argmax((OL.softmax(tgt_logits) * atoms[None, None, :]).sum(-1, dtype=f32), -1)
    p = _softmax(tgt_logits[bi, a_star])
    base, lo, up = c51_bins(r, d, atoms, vmin, vmax, G)
    b64 = _d(base)
    keep = up < M
    rows = np.broadcast_to(bi[:, None] * M, (B, M))
    m = np.zeros(B * M); sm = np.zeros(B * M)
    np.add.at(m, (rows + lo).ravel(), (p * (up - b64)).ravel())
    np.add.at(m, (rows + up)[keep], (p * (b64 - lo))[keep])
    np.add.at(sm, (rows + lo).ravel(), p.ravel())
    np.add.at(sm, (rows + up)[keep], p[keep])
    m = m.reshape(B, M); sm = sm.reshape(B, M)
    l = _d(logits[bi, a])
    z = l - l.max(-1, keepdims=True)
    lse = np.log(np.exp(z).sum(-1, keepdims=True))
    logp = z - lse
    k = np.abs(z) + np.abs(lse) + 1.0            # error scale of logp_j (and relative error scale of exp(logp_j))
    n = np.full((B, M), 3 * M + 16)
    loss = R(-(m * logp).sum(-1), (sm * k).sum(-1), np.full(B, 3 * M + 16))
    sp = np.exp(logp)
    gv = np.zeros((B, A, M)); gs = np.zeros((B, A, M)); gn = np.zeros((B, A, M))
    gv[bi, a] = _d(w)[:, None] * (sp * m.sum(-1, keepdims=True) - m)
    gs[bi, a] = np.abs(_d(w))[:, None] * (sp * k * sm.sum(-1, keepdims=True) + sm)
    gn[bi, a] = n
    return {"loss": loss, "grad": R(gv, gs, gn), "target_prob": R(m, sm, n)}


def quantile(qa, T, tau, w):
    """agent.py:110-114 for the selected rows: qa [B,Nj] online quantiles, T [B,Ni] fp32 targets, tau [B,Nj] or [Nj],
    w [B].  Returns loss [B] and the gradient wrt qa [B,Nj]."""
    B, Nj = qa.shape
    Ni = T.shape[1]
    pos = qa[:, None, :] > T[:, :, None]                       # u = q - T > 0, decided on the fp32 values
    u = _d(qa)[:, None, :] - _d(T)[:, :, None]
    t = np.broadcast_to(_d(tau), (B, Nj))[:, None, :]
    wt = np.where(pos, 1.0 - t, t)
    au = np.abs(u)
    c = np.minimum(au, 1.0)
    h = c * (au - 0.5 * c)
    loss = R((wt * h).sum((1, 2)) / Ni, (wt * (h + c * au)).sum((1, 2)) / Ni, np.full(B, Ni + Nj + 8))
    wn = _d(w)[:, None] / Ni
    grad = R(wn * (wt * np.clip(u, -1.0, 1.0)).sum(1), np.abs(wn) * (wt * 2.0 * c).sum(1), np.full((B, Nj), Ni + 8))
    return {"loss": loss, "grad": grad}


def fraction(qh, qb, taus, w):
    """FQF fraction loss (agent.py:371-387) for the selected rows: qh [B,F] (q at tau_hat), qb [B,F-1] (q at the
    interior taus), taus [B,F+1].  Returns fraction_loss [B] and its gradient wrt taus [B,F+1] (w-weighted)."""
    B, F = qh.shape
    prev = np.concatenate((qh[:, :1], qb[:, :-1]), 1)
    nxt = np.concatenate((qb[:, 1:], qh[:, -1:]), 1)
    v1 = _d(qb) - _d(qh[:, :-1])
    v2 = _d(qb) - _d(qh[:, 1:])
    g = np.where(qb > prev, v1, -v1) + np.where(qb < nxt, v2, -v2)
    sg = np.abs(v1) + np.abs(v2)
    ti = _d(taus[:, 1:-1])
    gt = np.zeros((B, F + 1)); st = np.zeros((B, F + 1))
    gt[:, 1:-1] = _d(w)[:, None] * g
    st[:, 1:-1] = np.abs(_d(w))[:, None] * sg
    return {"fraction_loss": R((g * ti).sum(1), (sg * np.abs(ti)).sum(1), np.full(B, F + 8)),
            "grad_taus": R(gt, st, np.full((B, F + 1), 4))}


def priority(loss, eps, alpha):
    """(loss + eps)^alpha (replay.py:55-59) of the fp32 losses a kernel returned, in float64."""
    return (_d(loss) + float(f32(eps))) ** float(f32(alpha))
