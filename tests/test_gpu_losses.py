"""K4 parity on the GPU: the fused target/loss kernels, called through the C ABI, against (a) the
golden outputs of the unmodified reference and (b) the numpy oracle on larger seeded inputs.
Tolerance: 1e-5 RELATIVE in fp32 (north_star) with an explicit denominator floor -- tests/parity.py:
|got - ref| <= 1e-5 * max(|ref|, 1e-2 * max|ref|) -- no absolute ``atol``; argmax/indices exact.  The worst
relative error per quantity is recorded by tests/parity.py."""
import numpy as np
import pytest
import torch

from oracle import losses as OL
from tests import parity

pytestmark = pytest.mark.gpu


def dev(x, dtype=None):
    t = torch.as_tensor(np.ascontiguousarray(x)).cuda()
    return t if dtype is None else t.to(dtype)


def close(name, got, want, **kw):
    parity.close(name, got, want, **kw)


def common(g):
    gam = np.float32(float(g["discount"]) ** int(g["n_step"]))
    return dev(g["actions"]), dev(g["rewards"]), dev(g["terminals"]), dev(g["weights"]), float(gam)


def prio_of(loss, eps=0.01):
    return np.sqrt(np.asarray(loss, dtype=np.float32) + np.float32(eps))


@pytest.mark.parametrize("dq", ["single", "double"])
def test_dqn_golden(golden, dq):
    from agent0_b200 import losses as L
    g = golden(f"loss_dqn_{dq}")
    a, r, d, w, gam = common(g)
    mp = torch.ones(1, device="cuda")
    out = L.dqn_loss(dev(g["online_cur"]), dev(g["tgt_next"]), a, r, d, w, gam,
                     qsel=dev(g["qval_next"]) if dq == "double" else None, max_p=mp)
    close("dqn.loss[golden]", out.loss, g["loss"]); close("dqn.grad[golden]", out.grad, g["grad"])
    close("dqn.prio[golden]", out.prio, prio_of(g["loss"]))
    close("dqn.max_p[golden]", mp, [max(1.0, float(g["loss"].max()))])


def test_mdqn_golden(golden):
    from agent0_b200 import losses as L
    g = golden("loss_mdqn_single")
    a, r, d, w, gam = common(g)
    out = L.mdqn_loss(dev(g["online_cur"]), dev(g["tgt_next"]), dev(g["tgt_cur"]), a, r, d, w, gam,
                      tau=float(g["tau"]), lo=float(g["lo"]))
    close("mdqn.loss[golden]", out.loss, g["loss"]); close("mdqn.grad[golden]", out.grad, g["grad"])


@pytest.mark.parametrize("dq", ["single", "double"])
def test_c51_golden(golden, dq):
    from agent0_b200 import losses as L
    g = golden(f"loss_c51_{dq}")
    a, r, d, w, gam = common(g)
    out = L.c51_loss(dev(g["online_cur"]), dev(g["tgt_next"]), dev(g["atoms"]), a, r, d, w, gam,
                     float(g["vmin"]), float(g["vmax"]), qsel=dev(g["qval_next"]) if dq == "double" else None,
                     want_target_prob=True)
    close("c51.loss[golden]", out.loss, g["loss"]); close("c51.grad[golden]", out.grad, g["grad"])
    _, _, m = OL.c51(g["online_cur"], g["tgt_next"], g["qval_next"] if dq == "double" else None, g["actions"],
                     g["rewards"], g["terminals"], g["weights"], float(g["discount"]), int(g["n_step"]),
                     g["atoms"], float(g["vmin"]), float(g["vmax"]))
    close("c51.target_prob[golden]", out.target_prob, m)          # projected distributions


@pytest.mark.parametrize("dq", ["single", "double"])
def test_qr_golden(golden, dq):
    from agent0_b200 import losses as L
    g = golden(f"loss_qr_{dq}")
    a, r, d, w, gam = common(g)
    out = L.qr_loss(dev(g["online_cur"]), dev(g["tgt_next"]), a, r, d, w, gam,
                    qsel=dev(g["qval_next"]) if dq == "double" else None)
    close("qr.loss[golden]", out.loss, g["loss"]); close("qr.grad[golden]", out.grad, g["grad"])


@pytest.mark.parametrize("dq", ["single", "double"])
def test_iqn_golden(golden, dq):
    """single: the action-selection values come from the target net (agent.py:305-308); the fixture holds
    whichever ``qval`` the reference used, the kernel's rule is the same."""
    from agent0_b200 import losses as L
    g = golden(f"loss_iqn_{dq}")
    a, r, d, w, gam = common(g)
    out = L.iqn_loss(dev(g["q_cur"]), dev(g["taus_cur"]), dev(g["q_next"]), dev(g["qval_next"]), a, r, d, w, gam)
    close("iqn.loss[golden]", out.loss, g["loss"]); close("iqn.grad[golden]", out.grad, g["grad"])


@pytest.mark.parametrize("dq", ["single", "double"])
def test_fqf_golden(golden, dq):
    from agent0_b200 import losses as L
    g = golden(f"loss_fqf_{dq}")
    a, r, d, w, gam = common(g)
    out = L.fqf_loss(dev(g["q_hat"]), dev(g["taus"]), dev(g["taus_hat"]), dev(g["q_next"]), dev(g["q_bar"]),
                     dev(g["qval_next"]), a, r, d, w, gam)
    close("fqf.loss[golden]", out.loss, g["loss"]); close("fqf.grad[golden]", out.grad, g["grad"])
    close("fqf.fraction_loss[golden]", out.fraction_loss, g["fraction_loss"])
    close("fqf.grad_taus[golden]", out.grad_taus, g["grad_taus"])


# ------------------------------------------------------------------ larger seeded cases vs the oracle
def _batch(rng, B, A):
    a = rng.randint(0, A, B).astype(np.int64)
    r = rng.choice([-1.0, 0.0, 1.0, 2.5], B).astype(np.float32)
    d = (rng.rand(B) < 0.2).astype(np.float32)
    w = (rng.rand(B) + 0.05).astype(np.float32)
    return a, r, d, w


@pytest.mark.parametrize("B,A,double", [(512, 4, True), (512, 18, False), (33, 6, True), (1, 4, False)])
def test_dqn_mdqn_oracle(B, A, double):
    from agent0_b200 import losses as L
    rng = np.random.RandomState(B + A)
    a, r, d, w = _batch(rng, B, A)
    q, tn, tc, qs = [(rng.randn(B, A) * 3).astype(np.float32) for _ in range(4)]
    gam = float(np.float32(0.99 ** 3))
    out = L.dqn_loss(dev(q), dev(tn), dev(a), dev(r), dev(d), dev(w), gam, qsel=dev(qs) if double else None)
    loss, grad = OL.dqn(q, tn, qs if double else None, a, r, d, w, 0.99, 3)
    # the gradient is w * clamp(q - T): a difference of operands of magnitude max(|q|, |T|), which is its error scale
    opscale = float(max(np.abs(q).max(), np.abs(tn).max() + np.abs(r).max()) * w.max())
    close("dqn.loss", out.loss, loss); close("dqn.grad", out.grad, grad, scale=opscale)
    out = L.mdqn_loss(dev(q), dev(tn), dev(tc), dev(a), dev(r), dev(d), dev(w), gam, tau=0.03, lo=-1.0)
    loss, grad = OL.mdqn(q, tn, tc, a, r, d, w, 0.99, 3, 0.03, -1.0)
    close("mdqn.loss", out.loss, loss, scale=opscale ** 2 / 2); close("mdqn.grad", out.grad, grad, scale=opscale)


@pytest.mark.parametrize("B,A,M,double", [(512, 4, 51, True), (64, 18, 51, False), (32, 4, 101, False)])
def test_c51_oracle(B, A, M, double):
    from agent0_b200 import losses as L
    rng = np.random.RandomState(B + A + M)
    a, r, d, w = _batch(rng, B, A)
    r[:4] = [30.0, -30.0, 0.0, 10.0]        # clamps at vmax / vmin, and an exactly-integer base
    d[2] = 1.0
    lg, tg = [(rng.randn(B, A, M) * 3).astype(np.float32) for _ in range(2)]
    qs = (rng.randn(B, A) * 3).astype(np.float32)
    atoms = torch.linspace(-10, 10, M).numpy()
    out = L.c51_loss(dev(lg), dev(tg), dev(atoms), dev(a), dev(r), dev(d), dev(w), float(np.float32(0.99 ** 3)),
                     -10.0, 10.0, qsel=dev(qs) if double else None, want_target_prob=True)
    loss, grad, m = OL.c51(lg, tg, qs if double else None, a, r, d, w, 0.99, 3, atoms, -10.0, 10.0)
    close("c51.target_prob", out.target_prob, m)
    close("c51.loss", out.loss, loss); close("c51.grad", out.grad, grad)
    close("c51.target_prob.sum", out.target_prob.sum(-1), np.ones(B))


@pytest.mark.parametrize("sorted_form", [1, 2, 0], ids=["sorted_cta", "sorted_warp", "pairwise"])
@pytest.mark.parametrize("B,A,N,double", [(512, 4, 200, True), (16, 18, 200, False), (8, 4, 7, False), (64, 6, 256, True),
                                          (32, 4, 65, False), (40, 4, 129, True)])
def test_qr_oracle(B, A, N, double, sorted_form):
    """All evaluations of the pair sums -- the O(N log N) sorted-target kernels (one CTA per sample: the default
    above 64 quantiles; one warp per sample) and the O(N^2) pair loop -- against the pairwise numpy oracle, and the
    sorted kernels against their own specification (oracle.losses.huber_qr_sorted, float64 prefix sums)."""
    from agent0_b200 import _lib
    from agent0_b200 import losses as L
    A0_OPT_QH_SORTED = 10
    rng = np.random.RandomState(B + A + N)
    a, r, d, w = _batch(rng, B, A)
    q, tn = [(rng.randn(B, A, N) * 3).astype(np.float32) for _ in range(2)]
    if N >= 129:                         # ties and exact range boundaries: targets equal to q, q-1, q+1; repeated targets
        q[0] = np.round(q[0]); tn[0] = np.round(tn[0]); r[0] = 0.0; d[0] = 0.0
        tn[1, :, 1::2] = tn[1, :, 0:-1:2]
    qs = (rng.randn(B, A) * 3).astype(np.float32)
    _lib.check(_lib.load().a0_set_option(A0_OPT_QH_SORTED, sorted_form), "a0_set_option")
    try:
        out = L.qr_loss(dev(q), dev(tn), dev(a), dev(r), dev(d), dev(w), float(np.float32(0.99 ** 3)),
                        qsel=dev(qs) if double else None)
        torch.cuda.synchronize()
    finally:
        _lib.check(_lib.load().a0_set_option(A0_OPT_QH_SORTED, 1), "a0_set_option")
    loss, grad = OL.qr(q, tn, qs if double else None, a, r, d, w, 0.99, 3)
    tag = ("pairwise", "sorted, CTA per sample", "sorted, warp per sample")[sorted_form] if N > 64 else "pairwise"
    close(f"qr.loss[{tag}]", out.loss, loss); close(f"qr.grad[{tag}]", out.grad, grad)
    if tag != "pairwise":
        bi = np.arange(B)
        a_star = np.argmax(qs, -1) if double else np.argmax(tn.mean(-1, dtype=np.float32), -1)
        T = OL._td_target(r[:, None], d[:, None], OL._G(0.99, 3), tn[bi, a_star])
        tau = ((2 * np.arange(N) + 1).astype(np.float32) / np.float32(2.0 * N)).astype(np.float32)
        l2, g2 = OL.huber_qr_sorted(q[bi, a], T, tau, w)
        close(f"qr.loss[{tag} vs its specification]", out.loss, l2)
        close(f"qr.grad[{tag} vs its specification]", out.grad.cpu().numpy()[bi, a], g2)


@pytest.mark.parametrize("B,A,N,Nd", [(512, 4, 64, 64), (8, 18, 64, 32), (5, 6, 8, 24)])
def test_iqn_oracle(B, A, N, Nd):
    from agent0_b200 import losses as L
    rng = np.random.RandomState(B + A + N + Nd)
    a, r, d, w = _batch(rng, B, A)
    q = (rng.randn(B, N, A) * 3).astype(np.float32)
    tn = (rng.randn(B, Nd, A) * 3).astype(np.float32)
    taus = rng.rand(B, N).astype(np.float32)
    qs = (rng.randn(B, A) * 3).astype(np.float32)
    out = L.iqn_loss(dev(q), dev(taus), dev(tn), dev(qs), dev(a), dev(r), dev(d), dev(w), float(np.float32(0.99 ** 3)))
    loss, grad = OL.iqn(q, taus, tn, qs, a, r, d, w, 0.99, 3)
    close("iqn.loss", out.loss, loss); close("iqn.grad", out.grad, grad)


@pytest.mark.parametrize("B,A,F", [(512, 4, 32), (9, 18, 32), (3, 4, 8)])
def test_fqf_oracle(B, A, F):
    from agent0_b200 import losses as L
    rng = np.random.RandomState(B + A + F)
    a, r, d, w = _batch(rng, B, A)
    qh = (rng.randn(B, F, A) * 3).astype(np.float32)
    tn = (rng.randn(B, F, A) * 3).astype(np.float32)
    qb = np.sort(rng.randn(B, F - 1, A) * 3, axis=1).astype(np.float32) + (rng.randn(B, F - 1, A) * 0.5).astype(np.float32)
    p = rng.rand(B, F).astype(np.float32) + 0.01
    p = p / p.sum(-1, keepdims=True)
    taus = np.concatenate((np.zeros((B, 1), np.float32), np.cumsum(p, -1).astype(np.float32)), axis=1)
    th = ((taus[:, :-1] + taus[:, 1:]) / 2).astype(np.float32)
    qs = (rng.randn(B, A) * 3).astype(np.float32)
    out = L.fqf_loss(dev(qh), dev(taus), dev(th), dev(tn), dev(qb), dev(qs), dev(a), dev(r), dev(d), dev(w),
                     float(np.float32(0.99 ** 3)))
    loss, grad, frac, gt = OL.fqf(qh, taus, th, tn, qb, qs, a, r, d, w, 0.99, 3)
    close("fqf.loss", out.loss, loss); close("fqf.grad", out.grad, grad)
    close("fqf.fraction_loss", out.fraction_loss, frac); close("fqf.grad_taus", out.grad_taus, gt)


def test_autograd_contract_matches_weighted_sum_backward():
    """online_out.backward(grad) must equal (loss*w).sum().backward() of the reference graph."""
    from agent0_b200 import losses as L
    torch.manual_seed(0)
    B, A = 64, 6
    lin = torch.nn.Linear(10, A).cuda()
    x = torch.randn(B, 10, device="cuda")
    tn = torch.randn(B, A, device="cuda") * 3
    a = torch.randint(0, A, (B,), device="cuda")
    r = torch.randn(B, device="cuda"); d = (torch.rand(B, device="cuda") < 0.2).float()
    w = torch.rand(B, device="cuda") + 0.1
    gam = float(np.float32(0.99))
    q = lin(x)
    out = L.dqn_loss(q, tn, a, r, d, w, gam)
    q.backward(out.grad)
    g_kernel = lin.weight.grad.clone(); lin.weight.grad = None
    q2 = lin(x)
    tgt = r + gam * (1 - d) * tn.max(-1)[0]
    loss = torch.nn.functional.smooth_l1_loss(q2[torch.arange(B), a], tgt, reduction="none")
    (loss * w).sum().backward()
    close("autograd.weight_grad (two fp32 GEMM orders)", g_kernel, lin.weight.grad.cpu().numpy(), rtol=1e-4)
    close("autograd.loss", out.loss, loss.detach().cpu().numpy())
