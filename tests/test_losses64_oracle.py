"""The float64 reference of the target/loss rules (oracle/losses64.py) against the fp32 oracle (oracle/losses.py) and
the golden outputs of the unmodified reference, the C51 rule for a base that rounds above M - 1, and the centred
prefix sums of the sorted quantile form against an exact pairwise float64 sum.  CPU only."""
import numpy as np
import pytest

from oracle import losses as OL
from oracle import losses64 as O64
from tests import parity

f32 = np.float32
EPS = 2.0 ** -24


def within_bound(name, got, r, slack=16):
    """|got - v| <= (n + slack) * 2^-24 * s per element (s = 0: exactly 0)."""
    err = np.abs(np.asarray(got, dtype=np.float64) - r.v)
    tol = (r.n + slack) * EPS * r.s
    bad = err > tol
    assert not bad.any(), f"{name}: {bad.sum()} elements outside the float64 bound, worst err/tol {np.max(err / np.maximum(tol, 1e-300)):.3g}"


def _gold_common(g):
    return g["actions"], g["rewards"], g["terminals"], g["weights"], OL._G(float(g["discount"]), int(g["n_step"]))


@pytest.mark.parametrize("dq", ["single", "double"])
def test_float64_reference_matches_the_golden_dqn_c51_qr(golden, dq):
    g = golden(f"loss_dqn_{dq}")
    a, r, d, w, G = _gold_common(g)
    o = O64.dqn(g["online_cur"], g["tgt_next"], g["qval_next"] if dq == "double" else None, a, r, d, w, G)
    parity.close("losses64.dqn.loss[golden]", o["loss"].v, g["loss"]); parity.close("losses64.dqn.grad[golden]", o["grad"].v, g["grad"])
    g = golden(f"loss_c51_{dq}")
    a, r, d, w, G = _gold_common(g)
    o = O64.c51(g["online_cur"], g["tgt_next"], g["qval_next"] if dq == "double" else None, a, r, d, w, G, g["atoms"],
                float(g["vmin"]), float(g["vmax"]))
    parity.close("losses64.c51.loss[golden]", o["loss"].v, g["loss"]); parity.close("losses64.c51.grad[golden]", o["grad"].v, g["grad"])
    g = golden(f"loss_qr_{dq}")
    a, r, d, w, G = _gold_common(g)
    q, tn = g["online_cur"], g["tgt_next"]
    B, _, N = q.shape
    bi = np.arange(B)
    a_star = np.argmax(g["qval_next"], -1) if dq == "double" else np.argmax(tn.mean(-1, dtype=f32), -1)
    T = OL._td_target(r[:, None], d[:, None], G, tn[bi, a_star])
    tau = ((2 * np.arange(N) + 1).astype(f32) / f32(2.0 * N)).astype(f32)
    o = O64.quantile(q[bi, a], T, tau, w)
    parity.close("losses64.qr.loss[golden]", o["loss"].v, g["loss"]); parity.close("losses64.qr.grad[golden]", o["grad"].v, g["grad"][bi, a])


def test_float64_reference_matches_the_golden_mdqn_iqn_fqf(golden):
    g = golden("loss_mdqn_single")
    a, r, d, w, G = _gold_common(g)
    o = O64.mdqn(g["online_cur"], g["tgt_next"], g["tgt_cur"], a, r, d, w, G, float(g["tau"]), float(g["lo"]))
    parity.close("losses64.mdqn.loss[golden]", o["loss"].v, g["loss"]); parity.close("losses64.mdqn.grad[golden]", o["grad"].v, g["grad"])
    for dq in ("single", "double"):
        g = golden(f"loss_iqn_{dq}")
        a, r, d, w, G = _gold_common(g)
        bi = np.arange(len(a))
        T = OL._td_target(r[:, None], d[:, None], G, g["q_next"][bi, :, np.argmax(g["qval_next"], -1)])
        o = O64.quantile(g["q_cur"][bi, :, a], T, g["taus_cur"].reshape(len(a), -1), w)
        parity.close("losses64.iqn.loss[golden]", o["loss"].v, g["loss"])
        parity.close("losses64.iqn.grad[golden]", o["grad"].v, g["grad"][bi, :, a])
        g = golden(f"loss_fqf_{dq}")
        a, r, d, w, G = _gold_common(g)
        o = O64.fraction(g["q_hat"][bi, :, a], g["q_bar"][bi, :, a], g["taus"], w)
        parity.close("losses64.fqf.fraction_loss[golden]", o["fraction_loss"].v, g["fraction_loss"])
        parity.close("losses64.fqf.grad_taus[golden]", o["grad_taus"].v, g["grad_taus"])


def _batch(rng, B, A):
    a = rng.randint(0, A, B).astype(np.int64)
    r = rng.choice([-1.0, 0.0, 1.0, 2.5, 30.0, -30.0], B).astype(f32)
    d = (rng.rand(B) < 0.2).astype(f32)
    w = (rng.rand(B) + 0.05).astype(f32)
    return a, r, d, w


@pytest.mark.parametrize("A", [1, 2, 7, 32])
def test_fp32_oracle_is_within_the_float64_bound_dqn_mdqn(A):
    """oracle/losses.py is one fp32 evaluation of the rules: it must lie within the error scale losses64 states."""
    rng = np.random.RandomState(A)
    B = 300
    a, r, d, w = _batch(rng, B, A)
    q, tn, tc, qs = [(rng.randn(B, A) * 3).astype(f32) for _ in range(4)]
    tn[:50] *= 27                                   # spreads of +-80: the softmax underflows
    qs[::4] = np.round(qs[::4])
    for G, dq in ((OL._G(0.99, 3), True), (f32(0), False), (f32(1), True)):
        o = O64.dqn(q, tn, qs if dq else None, a, r, d, w, G)
        loss, grad = OL.dqn(q, tn, qs if dq else None, a, r, d, w, float(G), 1)
        within_bound("dqn.loss", loss, o["loss"]); within_bound("dqn.grad", grad, o["grad"])
    for tau in (0.03, 1e-3):
        o = O64.mdqn(q, tn, tc, a, r, d, w, OL._G(0.99, 3), tau, -1.0)
        loss, grad = OL.mdqn(q, tn, tc, a, r, d, w, 0.99, 3, tau, -1.0)
        within_bound(f"mdqn.loss tau={tau}", loss, o["loss"]); within_bound(f"mdqn.grad tau={tau}", grad, o["grad"])
        parity.close("losses64.mdqn.loss", o["loss"].v, loss, scale=float(o["loss"].s.max()))


@pytest.mark.parametrize("M,vmin,vmax", [(51, -10.0, 10.0), (101, -10.0, 10.0), (128, -10.0, 10.0), (64, -5.0, 12.0),
                                         (33, -1.0, 50.0)])
def test_fp32_oracle_is_within_the_float64_bound_c51(M, vmin, vmax):
    rng = np.random.RandomState(M)
    B, A = 40, 5
    a, r, d, w = _batch(rng, B, A)
    lg, tg = [(rng.randn(B, A, M) * 3).astype(f32) for _ in range(2)]
    tg[0] = -200.0; tg[0, :, 3] = 0.0               # one-hot target distribution: exact zeros in fp32
    qs = (rng.randn(B, A) * 3).astype(f32)
    atoms = np.linspace(vmin, vmax, M).astype(f32)
    G = OL._G(0.99, 3)
    for sel in (qs, None):
        o = O64.c51(lg, tg, sel, a, r, d, w, G, atoms, vmin, vmax)
        loss, grad, m = OL.c51(lg, tg, sel, a, r, d, w, float(G), 1, atoms, vmin, vmax)
        tiny = 2.0 ** -126                          # terms that underflow in fp32
        for name, got in (("loss", loss), ("grad", grad), ("target_prob", m)):
            rr = o[name]
            within_bound(f"c51.{name}", got, O64.R(rr.v, rr.s + tiny * 2 ** 24, rr.n))
            parity.close(f"losses64.c51.{name}", rr.v, got)


# the supports for which fl32(fl32(vmax - vmin) / (M - 1)) puts the base of an atom clamped at vmax above M - 1
OVERFLOWING = [(128, -10.0, 25.0), (128, -10.0, 7.0), (128, -5.0, 12.0), (128, -1.0, 50.0), (128, -1.0, 0.7),
               (51, -10.0, 200.0), (101, -10.0, 200.0), (51, -5.0, 100.0), (101, -5.0, 100.0), (64, -10.0, 0.7),
               (124, -10.0, 10.0)]


@pytest.mark.parametrize("M,vmin,vmax", OVERFLOWING)
def test_c51_base_above_the_last_bin_drops_the_upper_term(M, vmin, vmax):
    """The kernels' fp32 bin arithmetic gives up == M for an atom clamped at vmax on these supports.  The projection
    drops that term (a0_k4_c51_fast always has; a0_k4_c51 wrote it past the sample's row), and the fp32 oracle does
    the same instead of raising IndexError."""
    atoms = np.linspace(vmin, vmax, M).astype(f32)
    r = np.array([1000.0, 0.0], f32); d = np.array([1.0, 0.0], f32)     # every atom clamped at vmax; a spread return
    base, lo, up = O64.c51_bins(r, d, atoms, vmin, vmax, f32(0.99))
    assert (up[0] == M).all() and (lo[0] == M - 1).all() and (base[0] > M - 1).all()
    p = np.full((2, M), 1.0 / M, f32)
    o = O64.c51(np.zeros((2, 1, M), f32), np.zeros((2, 1, M), f32), None, np.zeros(2, np.int64), r, d,
                np.ones(2, f32), f32(0.99), atoms, vmin, vmax)
    v = o["target_prob"].v[0]
    assert (v[:M - 1] == 0).all() and v[M - 1] < 1.0
    np.testing.assert_allclose(v[M - 1], (np.float64(1.0 / M) * (M - base[0].astype(np.float64))).sum(), rtol=1e-12)
    m = OL.c51_project(p, r, d, atoms, vmin, vmax, f32(0.99))
    # The reference's delta is fl32 of a float64 division; it equals the kernels' where vmax - vmin is exact in fp32
    # (with vmax = 0.7 the two deltas differ in the last bit, and the oracle's base stays below M - 1)
    if float(f32(f32(vmax) - f32(vmin))) == vmax - vmin:
        parity.close("losses64.c51.target_prob[base above M-1]", v[None], m[:1])
        assert (m[0, :M - 1] == 0).all()
        np.testing.assert_allclose(m[0, M - 1], (p[0] * (f32(M) - base[0])).sum(dtype=np.float64), rtol=1e-6)


@pytest.mark.parametrize("c", [0.0, 1e3, 1e4, 1e5, 1e6])
def test_sorted_quantile_form_is_centred(c):
    """oracle.losses.huber_qr_sorted (the specification of the sorted K4 kernels) against the exact pairwise float64
    sums at large offsets.  Without the centring of its prefix sums the loss is 8e-5 off at 1e5 and 8e-3 at 1e6."""
    rng = np.random.RandomState(int(c) % 1000)
    B, N = 6, 200
    q = (c + 0.4 * rng.randn(B, N)).astype(f32)
    T = (c + 0.4 * rng.randn(B, N)).astype(f32)
    T[0, ::3] = q[0, ::3]; T[1] = T[1, 0]                   # targets equal to q; all targets equal
    tau = ((2 * np.arange(N) + 1).astype(f32) / f32(2.0 * N)).astype(f32)
    w = (rng.rand(B) + 0.1).astype(f32)
    loss, grad = OL.huber_qr_sorted(q, T, tau, w)
    o = O64.quantile(q, T, tau, w)
    parity.close(f"huber_qr_sorted.loss[offset {c:g}]", loss, o["loss"].v, rtol=1e-6)
    parity.close(f"huber_qr_sorted.grad[offset {c:g}]", grad, o["grad"].v, rtol=1e-6)


@pytest.mark.parametrize("Ni,Nj", [(1, 1), (1, 64), (64, 1), (65, 256), (200, 128)])
def test_fp32_oracle_is_within_the_float64_bound_quantile_and_fraction(Ni, Nj):
    rng = np.random.RandomState(Ni * 7 + Nj)
    B = 5
    q = (rng.randn(B, Nj) * 3).astype(f32)
    T = (rng.randn(B, Ni) * 3).astype(f32)
    T[0] = np.round(T[0]); q[0] = np.round(q[0])           # ties and exact range boundaries
    tau = rng.rand(B, Nj).astype(f32); tau[0, ::2] = 0.0; tau[1, ::2] = 1.0
    w = (rng.rand(B) + 0.1).astype(f32)
    o = O64.quantile(q, T, tau, w)
    loss = OL.huber_qr_loss(q[:, None, :], T[:, :, None], tau[:, None, :])
    grad = OL._huber_qr_grad(q, T, tau, w)
    within_bound("quantile.loss", loss, o["loss"]); within_bound("quantile.grad", grad, o["grad"])
    if Ni == Nj and Ni >= 2:
        F = Ni
        qb = (rng.randn(B, F - 1) * 3).astype(f32); qb[0, ::2] = q[0, 1::2][:len(qb[0, ::2])]
        p = rng.rand(B, F).astype(f32) + 0.01
        taus = np.concatenate((np.zeros((B, 1), f32), np.cumsum(p / p.sum(-1, keepdims=True), -1).astype(f32)), 1)
        fo = O64.fraction(q, qb, taus, w)
        a = np.zeros(B, np.int64)
        _, _, frac, gt = OL.fqf(q[:, :, None], taus, taus[:, 1:], T[:, :, None], qb[:, :, None], np.zeros((B, 1), f32), a,
                                np.zeros(B, f32), np.ones(B, f32), w, 0.99, 1)
        within_bound("fraction_loss", frac, fo["fraction_loss"]); within_bound("grad_taus", gt, fo["grad_taus"])
