"""Every K4 dispatch path across the shapes the C ABI accepts, against the fp32 oracle and a float64 evaluation.

The target/loss entry points choose among eleven kernel instantiations by A, M, Ni, Nj, the layout and qsel.  Each case
calls the C ABI directly, with every output buffer pre-filled with NaN (an element a kernel fails to write is caught),
and checks
  (a) the 1e-5 contract against oracle/losses.py (tests/parity.py; the C51 gradient against the float64 value);
  (b) |got - v64| <= (n + 16) * 2^-24 * s64 per element against oracle/losses64.py, so that a kernel and the fp32
      oracle cannot share an error; an element with s64 = 0 (outside the taken action's row or column) must be 0;
  (c) max_p equal to the largest finite loss and the priorities equal to the float64 (loss + eps)^alpha to 1e-5;
  (d) two launches bit-identical (a race shows up here);
  (e) bit-identity between the paths that are the same arithmetic: a0_k4_c51_fast and a0_k4_c51 (A0_OPT_C51_FAST),
      the quantile kernels with and without the all-action fetch (A0_OPT_QH_SPEC);
and the sorted quantile kernels against their specification oracle.losses.huber_qr_sorted to 1e-6.  Where a reference
value is NaN or infinite (a NaN selection value picks its action, as torch.argmax does, so its row's outputs are NaN),
the kernel's value must be the same."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import losses as OL
from oracle import losses64 as O64
from tests import parity

pytestmark = pytest.mark.gpu

f32 = np.float32
OPT_C51_FAST, OPT_QH_SORTED, OPT_QH_SPEC = 5, 10, 14        # include/agent0_b200.h
PRIO_EPS = 0.01
ALPHAS = (0.5, 0.6, 1.0)
G3 = float(f32(0.99 ** 3))
TINY = 2.0 ** -126          # absolute slack for terms that underflow in fp32 (softmax tails): only where s64 > 0


@pytest.fixture
def lib():
    from agent0_b200 import _lib
    L = _lib.load()
    yield L
    for opt in (OPT_C51_FAST, OPT_QH_SORTED, OPT_QH_SPEC):
        L.a0_set_option(opt, 1)


def _set(lib, opt, value):
    assert lib.a0_set_option(opt, value) == 0


def dev(x):
    return torch.as_tensor(np.ascontiguousarray(x)).cuda()


def launch(call, B, A, a, r, d, w, G, alpha, shapes):
    """One K4 launch through the C ABI into NaN-filled buffers (max_p starts at 0).  Returns numpy outputs."""
    from agent0_b200 import _lib
    bufs = {"loss": torch.full((B,), float("nan"), device="cuda"), "prio": torch.full((B,), float("nan"), device="cuda"),
            "max_p": torch.zeros(1, device="cuda")}
    bufs.update({k: torch.full(s, float("nan"), device="cuda") for k, s in shapes.items()})
    c = _lib.LossCommon(B=B, A=A, action=a.data_ptr(), reward=r.data_ptr(), done=d.data_ptr(), weight=w.data_ptr(), gamma_n=G,
                        alpha=alpha, eps=PRIO_EPS, loss=bufs["loss"].data_ptr(), prio=bufs["prio"].data_ptr(),
                        max_p=bufs["max_p"].data_ptr())
    _lib.check(call(C.byref(c), {k: v.data_ptr() for k, v in bufs.items()}, _lib.stream_ptr()), "K4 launch")
    torch.cuda.synchronize()
    return {k: v.cpu().numpy() for k, v in bufs.items()}


def launch_twice(*args):
    o1, o2 = launch(*args), launch(*args)
    for k in o1:
        assert np.array_equal(o1[k].view(np.uint32), o2[k].view(np.uint32)), f"{k}: two launches differ"
    return o1


def same_bits(name, x, y):
    for k in x:
        assert np.array_equal(x[k].view(np.uint32), y[k].view(np.uint32)), f"{name}: {k} differs"


def finite_part(name, got, want):
    """Where ``want`` is NaN or infinite, ``got`` must be the same (any NaN for NaN).  Returns the mask of the rest."""
    got, want = np.asarray(got), np.asarray(want)
    odd = ~np.isfinite(want) | ~np.isfinite(got)
    same = (np.isnan(got) & np.isnan(want)) | (got == want)
    bad = odd & ~same
    assert not bad.any(), (f"{name}: {int(bad.sum())} non-finite elements differ, e.g. index {np.argwhere(bad)[0].tolist()}: "
                           f"got {got[bad][0]!r}, reference {want[bad][0]!r}")
    return ~odd


def bound64(name, got, r):
    """(b) of the module docstring for one output against its losses64.R."""
    ok = finite_part(name, got, r.v)
    got = np.asarray(got, np.float64)
    err = np.abs(got - r.v)
    tol = (r.n + 16) * 2.0 ** -24 * r.s + np.where(r.s > 0, TINY, 0.0)
    bad = ok & ~(err <= tol)
    assert not bad.any(), (f"{name}: {int(bad.sum())} elements outside the float64 bound, e.g. index "
                           f"{np.argwhere(bad)[0].tolist()}: got {got[bad][0]!r}, float64 {r.v[bad][0]!r}, bound {tol[bad][0]:.3g}")


def check(name, out, ref32, ref64, alpha, scales=None):
    """(a), (b) and (c) of the module docstring.  ref32: {key: fp32 oracle}; ref64: {key: losses64.R}."""
    for k, r in ref64.items():
        bound64(f"{name}.{k}", out[k], r)
    for k, want in ref32.items():
        ok = finite_part(f"{name}.{k}", out[k], want)
        parity.close(f"{name}.{k}", out[k][ok], want[ok], scale=(scales or {}).get(k))
    loss = out["loss"]
    fin = loss[np.isfinite(loss)]
    assert out["max_p"][0] == max(0.0, float(fin.max()) if fin.size else 0.0), f"{name}: max_p"
    prio = O64.priority(loss, PRIO_EPS, alpha)
    ok = finite_part(f"{name}.prio", out["prio"], prio)
    parity.close(f"{name}.prio[alpha={alpha}]", out["prio"][ok], prio[ok])


def nan_selection_rows(A):
    """Selection values (qsel) whose arg-max depends on NaN being the largest value, the first NaN winning: NaN first, in
    the middle, last; the row a '>' butterfly split three ways; all NaN; NaN next to +inf."""
    n, inf = f32(np.nan), f32(np.inf)
    base = np.linspace(-1.0, 1.0, A, dtype=f32)
    rows = []
    for j in (0, A // 2, A - 1):
        r = base.copy(); r[j] = n; rows.append(r)
    r = np.full(A, -2.0, f32); r[:4] = [1.0, n, 5.0, 9.0][:A]; rows.append(r)
    rows.append(np.full(A, n, f32))
    r = base.copy(); r[max(A - 2, 0)] = inf; r[A - 1] = n; rows.append(r)
    return rows


def put_rows(x, rows, start):
    """x[start + i] = rows[i] where x has room."""
    for i, row in enumerate(rows[:max(0, len(x) - start)]):
        x[start + i] = row


def _batch(rng, B, A, rewards=(-1.0, 0.0, 1.0, 2.5)):
    a = rng.randint(0, A, B).astype(np.int64)
    r = rng.choice(rewards, B).astype(f32)
    d = (rng.rand(B) < 0.25).astype(f32)
    w = (rng.rand(B) + 0.05).astype(f32)
    return a, r, d, w


# ---------------------------------------------------------------------------------------------------- DQN / M-DQN
@pytest.mark.parametrize("B", [1, 3, 4, 5, 1000])
@pytest.mark.parametrize("A", [1, 2, 31, 32])
def test_dqn_and_mdqn(lib, A, B):
    """a0_k4_dqn in both modes: exact ties (first index wins), spreads of +-80 (the softmax underflows), tau 0.03 and
    1e-3, terminal transitions, gamma^n in {0, 1}."""
    rng = np.random.RandomState(100 * A + B)
    a, r, d, w = _batch(rng, B, A)
    d[0] = 1.0
    q, tn, tc, qs = [(rng.randn(B, A) * 3).astype(f32) for _ in range(4)]
    tn[1::4] *= 27; tc[2::4] *= 27; q[3::4] *= 27
    qs[::2] = np.round(qs[::2] / 3); tn[::5] = np.round(tn[::5] / 3)
    put_rows(qs, nan_selection_rows(A), 7)          # B = 1000: each target row has distinct values, so a* shows
    ag, rg, dg, wg, qg, tng, tcg, qsg = map(dev, (a, r, d, w, q, tn, tc, qs))
    # the gradient w * clamp(q - T) is a difference of operands of magnitude max(|q|, |T|), which is its error scale
    sc = float(max(np.abs(q).max(), np.abs(tn).max() + np.abs(r).max() + 1.0) * w.max())
    for i, (G, dq) in enumerate(((G3, True), (0.0, False), (1.0, True), (G3, False))):
        alpha = ALPHAS[i % 3]
        out = launch_twice(lambda c, o, s: lib.a0_loss_dqn(c, qg.data_ptr(), tng.data_ptr(), qsg.data_ptr() if dq else None,
                                                           o["grad"], s), B, A, ag, rg, dg, wg, G, alpha, {"grad": (B, A)})
        loss, grad = OL.dqn(q, tn, qs if dq else None, a, r, d, w, G, 1)
        check(f"shapes.dqn[A={A}]", out, {"loss": loss, "grad": grad},
              O64.dqn(q, tn, qs if dq else None, a, r, d, w, G), alpha, {"grad": sc})
    for i, tau in enumerate((0.03, 1e-3)):
        alpha = ALPHAS[(i + 1) % 3]
        out = launch_twice(lambda c, o, s: lib.a0_loss_mdqn(c, qg.data_ptr(), tng.data_ptr(), tcg.data_ptr(), tau, -1.0, o["grad"], s),
                           B, A, ag, rg, dg, wg, G3, alpha, {"grad": (B, A)})
        loss, grad = OL.mdqn(q, tn, tc, a, r, d, w, G3, 1, tau, -1.0)
        check(f"shapes.mdqn[A={A},tau={tau}]", out, {"loss": loss, "grad": grad},
              O64.mdqn(q, tn, tc, a, r, d, w, G3, tau, -1.0), alpha, {"loss": sc * sc / 2, "grad": sc})


# ---------------------------------------------------------------------------------------------------- C51
# symmetric and asymmetric supports; most put the base of an atom clamped at vmax above M - 1 for some M (the symmetric
# one at M = 124; tests/test_losses64_oracle.py): that upper term is dropped
SUPPORTS = [(-10.0, 10.0), (-5.0, 12.0), (-10.0, 25.0), (-10.0, 7.0), (-1.0, 50.0), (-1.0, 0.7), (-10.0, 200.0),
            (-5.0, 100.0), (-10.0, 0.7)]


def _c51_inputs(M, A, B, vmin, vmax, seed):
    rng = np.random.RandomState(seed)
    a, r, d, w = _batch(rng, B, A, rewards=(-1.0, 0.0, 1.0, 9.99, -30.0, 30.0, 0.4, 2.0))
    atoms = np.linspace(vmin, vmax, M).astype(f32)
    r[0], d[0] = 1000.0, 0.0                   # every atom clamped at vmax
    r[1], d[1] = -1000.0, 0.0                  # ... at vmin
    r[2], d[2] = 0.5, 1.0                      # terminal: all mass to one or two bins
    r[3], d[3] = atoms[M // 2], 1.0            # an (almost) integer base
    lg, tg = [(rng.randn(B, A, M) * 3).astype(f32) for _ in range(2)]
    tg[4] = -200.0; tg[4, :, 1] = 0.0          # one-hot target logits: exact zeros in p
    qs = (rng.randn(B, A) * 3).astype(f32)
    qs[5] = 1.0                                # ties: the first maximum wins
    put_rows(qs, nan_selection_rows(A), 6)     # NaN selection values: samples 6-11
    tg[12, A - 1, M // 3] = np.nan             # without qsel the last action's expected value is NaN: it is selected
    return a, r, d, w, atoms, lg, tg, qs


def _c51_case(lib, M, A, B, vmin, vmax, qsel, fast_too, seed):
    a, r, d, w, atoms, lg, tg, qs = _c51_inputs(M, A, B, vmin, vmax, seed)
    ag, rg, dg, wg, lgg, tgg, qsg, atg = map(dev, (a, r, d, w, lg, tg, qs, atoms))
    sel = qs if qsel else None
    alpha = ALPHAS[seed % 3]

    def call(c, o, s):
        return lib.a0_loss_c51(c, lgg.data_ptr(), tgg.data_ptr(), qsg.data_ptr() if qsel else None, atg.data_ptr(), M, vmin, vmax,
                               o["grad"], o["target_prob"], s)
    args = (call, B, A, ag, rg, dg, wg, G3, alpha, {"grad": (B, A, M), "target_prob": (B, M)})
    _set(lib, OPT_C51_FAST, 0)
    out = launch_twice(*args)
    _set(lib, OPT_C51_FAST, 1)
    if fast_too:
        same_bits(f"c51 fast vs general M={M} A={A} ({vmin},{vmax})", launch_twice(*args), out)
    tag = f"shapes.c51[M={M},A={A},({vmin:g},{vmax:g})]"
    ref64 = O64.c51(lg, tg, sel, a, r, d, w, G3, atoms, vmin, vmax)
    # the gradient w * (p_j * sum(m) - m_j) is a difference of operands of size up to w, which is its error scale, and
    # each operand carries its own softmax rounding: at M = 2 and 3 (terms ~0.8, difference ~2e-3) the fp32 oracle alone
    # is up to 9e-6 off the float64 value under this scale (2.6e-5 under the default floor), so the gradient is held to
    # the contract against the float64 value
    wm = np.abs(w)[:, None] * ref64["target_prob"].v
    sc = float(np.nanmax(np.abs(ref64["grad"].v[np.arange(B), a] + wm) + wm))   # NaN rows: the NaN-selection samples
    ref32 = {"grad": ref64["grad"].v}
    # the reference's delta is fl32 of a float64 division, the kernels' an fp32 division of fl32(vmax - vmin): where the two
    # differ in the last bit (vmax = 0.7) so do the bins, and only the float64 evaluation of the kernels' rule applies
    if f32((vmax - vmin) / (M - 1)) == f32(f32(f32(vmax) - f32(vmin)) / f32(M - 1)):
        loss, _, m = OL.c51(lg, tg, sel, a, r, d, w, G3, 1, atoms, vmin, vmax)
        ref32.update(loss=loss, target_prob=m)
    check(tag, out, ref32, ref64, alpha, {"grad": sc})
    tp = out["target_prob"]
    tp = tp[np.isfinite(tp).all(-1)]              # the NaN rows were matched to the references above
    assert (tp.sum(-1) <= 1.0 + 1e-5).all()


@pytest.mark.parametrize("A", [1, 5, 6])
@pytest.mark.parametrize("M", [2, 3, 31, 32, 33, 63, 64])
def test_c51_fast_eligible_shapes(lib, M, A):
    """qsel given, A <= 6, M <= 64: a0_k4_c51_fast bit-identical to a0_k4_c51; without qsel the general kernel's
    arg-max over expected values.  B = 13: the last CTA of four samples is partial."""
    for i, (vmin, vmax) in enumerate(SUPPORTS):
        _c51_case(lib, M, A, 13, vmin, vmax, True, True, M * 31 + A * 7 + i)
        if i < 3:
            _c51_case(lib, M, A, 13, vmin, vmax, False, False, M * 31 + A * 7 + i)


@pytest.mark.parametrize("A", [7, 18, 32])
@pytest.mark.parametrize("M", [65, 96, 97, 124, 127, 128])
def test_c51_general_kernel_shapes(lib, M, A):
    """a0_k4_c51 with three and four atoms per lane, up to 32 actions.  M = 128 with an overflowing support is the case
    whose upper term used to land in bin 0 of the next sample of the CTA; M = 124 overflows on the symmetric support."""
    for i, (vmin, vmax) in enumerate(SUPPORTS):
        _c51_case(lib, M, A, 13, vmin, vmax, i % 2 == 0, False, M * 31 + A * 7 + i)


# ---------------------------------------------------------------------------------------------------- quantile family
def _quantile_refs(q, qt, taus, qs, a, r, d, w, G, layout, Ni, Nj, qsel):
    """Selection (first maximum, on fp32 values), targets T and the per-sample rows; the oracle and float64 references
    laid out like the kernel's gradient."""
    B, A = qs.shape
    bi = np.arange(B)
    qv = q if layout == 0 else q.transpose(0, 2, 1)             # [B, A, N]
    tv = qt if layout == 0 else qt.transpose(0, 2, 1)
    a_star = np.argmax(qs, -1) if qsel else np.argmax(tv.mean(-1, dtype=f32), -1)
    T = OL._td_target(r[:, None], d[:, None], f32(G), tv[bi, a_star])
    qa = qv[bi, a]
    tau = taus if taus is not None else np.broadcast_to(((2 * np.arange(Nj) + 1).astype(f32) / f32(2.0 * Nj)).astype(f32), (B, Nj))
    loss = OL.huber_qr_loss(qa[:, None, :], T[:, :, None], tau[:, None, :])
    g32 = np.zeros((B, A, Nj), f32)
    g32[bi, a] = OL._huber_qr_grad(qa, T, tau, w)
    o64 = O64.quantile(qa, T, tau, w)
    gv, gs = np.zeros((B, A, Nj)), np.zeros((B, A, Nj))
    gv[bi, a], gs[bi, a] = o64["grad"].v, o64["grad"].s
    g = o64["grad"].n[0, 0]
    if layout == 1:
        g32, gv, gs = g32.transpose(0, 2, 1), gv.transpose(0, 2, 1), gs.transpose(0, 2, 1)
    return {"loss": loss, "grad": np.ascontiguousarray(g32)}, {"loss": o64["loss"], "grad": O64.R(gv, gs, g)}, qa, T, tau


def _quantile_inputs(rng, B, A, Ni, Nj, layout, c=0.0, spread=3.0):
    """q around c, target network outputs around 2c (T = r + 0.5 * boot, G = 0.5); sample 0 terminal (all targets equal
    r), sample 1 on the integer lattice (targets equal to q and q +- 1, repeated targets), sample 2 with the same target row
    for every action (ties in the mean-argmax), layout 1 with tau exactly 0 and 1 in places."""
    a, r, d, w = _batch(rng, B, A)
    d[:] = 0.0; d[0] = 1.0
    q = (c + spread * rng.randn(B, A, Nj)).astype(f32)
    qt = (2 * c + 2 * spread * rng.randn(B, A, Ni)).astype(f32)
    q[0, :, ::2] = r[0]; q[0, :, 1::4] = r[0] + 1.0
    r[1] = 0.0
    q[1] = np.round(q[1] - c) + f32(c)
    qt[1] = 2 * (np.round(qt[1] / 2 - c) + f32(c))
    if B > 2:
        qt[2] = qt[2, :1]
    qs = rng.randn(B, A).astype(f32)
    qs[1] = 0.0                                                  # tie: a* = 0
    if c:
        # at an offset the row means (the selection without qsel) carry a rounding error of up to Ni * 2^-24 * |2c|, more
        # than their spread, so any two fp32 summation orders may pick different rows: every row but the one qsel picks is
        # lowered by twice that bound.  Sample 2 keeps its equal rows (equal sums in any order: the first wins).
        margin = f32(2 * Ni * 2.0 ** -24 * abs(2 * c) + 8 * spread)
        for b in (b for b in range(B) if b != 2):
            qt[b, np.arange(A) != np.argmax(qs[b])] -= margin
    taus = None
    if layout == 1:
        q, qt = q.transpose(0, 2, 1).copy(), qt.transpose(0, 2, 1).copy()
        taus = rng.rand(B, Nj).astype(f32)
        taus[0, ::3] = 0.0; taus[1, ::3] = 1.0
    return a, r, d, w, q, qt, taus, qs


def _quantile_call(lib, layout, qg, qtg, tg, qsg, Ni, Nj):
    def call(c, o, s):
        return lib.a0_loss_quantile(c, layout, qg.data_ptr(), qtg.data_ptr(), tg.data_ptr() if tg is not None else None,
                                    qsg.data_ptr() if qsg is not None else None, Ni, Nj, o["grad"], None, None, None, None, s)
    return call


@pytest.mark.parametrize("layout,qsel", [(0, False), (0, True), (1, True)], ids=["qr", "qr_qsel", "iqn"])
@pytest.mark.parametrize("A", [1, 8, 9, 32])
@pytest.mark.parametrize("Ni,Nj", [(1, 1), (1, 64), (64, 1), (32, 64), (64, 200), (200, 64), (256, 32)])
def test_quantile_pair_loop(lib, Ni, Nj, A, layout, qsel):
    """a0_k4_quantile<true | false>: at most 64 targets or at most 64 online quantiles, Ni != Nj, up to 256 threads."""
    rng = np.random.RandomState(Ni * 1000 + Nj * 10 + A + layout)
    B, G = 12, 0.5
    a, r, d, w, q, qt, taus, qs = _quantile_inputs(rng, B, A, Ni, Nj, layout)
    put_rows(qs, nan_selection_rows(A), B - 6)                   # NaN selection values: the last six samples
    if not qsel:
        # the last action's row mean is NaN (+inf and -inf targets): it is selected and the targets are +-inf
        qt[B - 1, A - 1, 0] = np.inf
        qt[B - 1, A - 1, Ni - 1] = -np.inf if Ni > 1 else np.inf
    ag, rg, dg, wg, qg, qtg, qsg = map(dev, (a, r, d, w, q, qt, qs))
    tg = dev(taus) if taus is not None else None
    alpha = ALPHAS[(Ni + Nj + A) % 3]
    gshape = (B, A, Nj) if layout == 0 else (B, Nj, A)
    args = (_quantile_call(lib, layout, qg, qtg, tg, qsg if qsel else None, Ni, Nj), B, A, ag, rg, dg, wg, G, alpha, {"grad": gshape})
    out = launch_twice(*args)
    _set(lib, OPT_QH_SPEC, 0)
    same_bits(f"quantile all-action fetch on/off Ni={Ni} Nj={Nj} A={A}", launch_twice(*args), out)
    _set(lib, OPT_QH_SPEC, 1)
    ref32, ref64, *_ = _quantile_refs(q, qt, taus, qs, a, r, d, w, G, layout, Ni, Nj, qsel)
    check(f"shapes.quantile_pairs[{Ni}x{Nj},A={A},layout={layout}]", out, ref32, ref64, alpha)


@pytest.mark.parametrize("layout,qsel", [(0, False), (0, True), (1, True)], ids=["qr", "qr_qsel", "iqn"])
@pytest.mark.parametrize("A", [4, 5, 8, 9])
@pytest.mark.parametrize("Ni,Nj", [(65, 65), (65, 256), (256, 65), (255, 255), (256, 256), (200, 128)])
def test_quantile_sorted_forms(lib, Ni, Nj, A, layout, qsel):
    """a0_k4_quantile_sorted<true,4>, <true,8>, <false,1> and a0_k4_quantile_warp, QR and IQN (layout 1, per-sample tau),
    with the quantiles offset by up to 1e6: the float64 prefix sums must stay within the contract at any magnitude."""
    G = 0.5
    for k, c in enumerate((0.0, 1e3, 1e5, 1e6)):
        rng = np.random.RandomState(Ni * 1000 + Nj * 10 + A + layout + k)
        a, r, d, w, q, qt, taus, qs = _quantile_inputs(rng, 4, A, Ni, Nj, layout, c=c, spread=2.0)
        if k == 0:
            # six more samples with NaN selection values
            more = _quantile_inputs(np.random.RandomState(Ni * 1000 + Nj * 10 + A + layout + 99), 6, A, Ni, Nj, layout)
            put_rows(more[-1], nan_selection_rows(A), 0)
            a, r, d, w, q, qt, taus, qs = [None if x is None else np.concatenate((x, y)) for x, y in zip((a, r, d, w, q, qt, taus, qs), more)]
        B = len(a)
        gshape = (B, A, Nj) if layout == 0 else (B, Nj, A)
        ag, rg, dg, wg, qg, qtg, qsg = map(dev, (a, r, d, w, q, qt, qs))
        tg = dev(taus) if taus is not None else None
        alpha = ALPHAS[k % 3]
        args = (_quantile_call(lib, layout, qg, qtg, tg, qsg if qsel else None, Ni, Nj), B, A, ag, rg, dg, wg, G, alpha, {"grad": gshape})
        out = launch_twice(*args)
        _set(lib, OPT_QH_SPEC, 0)
        same_bits(f"sorted all-action fetch on/off Ni={Ni} Nj={Nj} A={A} c={c:g}", launch_twice(*args), out)
        _set(lib, OPT_QH_SPEC, 1)
        _set(lib, OPT_QH_SORTED, 2)
        warp = launch_twice(*args)
        _set(lib, OPT_QH_SORTED, 1)
        ref32, ref64, qa, T, tau = _quantile_refs(q, qt, taus, qs, a, r, d, w, G, layout, Ni, Nj, qsel)
        l_spec, g_spec = OL.huber_qr_sorted(qa, T, tau, w)
        bi = np.arange(B)
        for form, o in (("cta", out), ("warp", warp)):
            tag = f"shapes.quantile_sorted_{form}[{Ni}x{Nj},A={A},layout={layout},c={c:g}]"
            check(tag, o, ref32, ref64, alpha)
            parity.close(f"{tag}.loss vs its specification", o["loss"], l_spec, rtol=1e-6)
            g = o["grad"][bi, a] if layout == 0 else o["grad"][bi, :, a]
            parity.close(f"{tag}.grad vs its specification", g, g_spec, rtol=1e-6)


@pytest.mark.parametrize("A", [1, 8, 9])
@pytest.mark.parametrize("F", [2, 3, 33, 64, 65, 256])
def test_fqf_fraction_term(lib, F, A):
    """The pair loop with the FQF fraction loss and its gradient wrt tau, with neighbouring q-bar and q-hat equal (the
    strict comparisons of agent.py:371-387)."""
    rng = np.random.RandomState(F * 10 + A)
    B, G = 5, G3
    a, r, d, w = _batch(rng, B, A)
    qh = (rng.randn(B, F, A) * 3).astype(f32)
    tn = (rng.randn(B, F, A) * 3).astype(f32)
    qb = (np.sort(rng.randn(B, F - 1, A) * 3, axis=1) + rng.randn(B, F - 1, A) * 0.5).astype(f32)
    qb[0, ::2] = qh[0, :F - 1:2]                     # q-bar equal to the q-hat on its left
    qb[1, 1::2] = qh[1, 2::2]                        # ... on its right
    qb[2, 1:] = qb[2, :-1]                           # equal q-bar neighbours
    p = rng.rand(B, F).astype(f32) + 0.01
    taus = np.concatenate((np.zeros((B, 1), f32), np.cumsum(p / p.sum(-1, keepdims=True), -1).astype(f32)), 1)
    th = ((taus[:, :-1] + taus[:, 1:]) / 2).astype(f32)
    qs = (rng.randn(B, A) * 3).astype(f32)
    ag, rg, dg, wg, qhg, tng, qbg, tg, thg, qsg = map(dev, (a, r, d, w, qh, tn, qb, taus, th, qs))
    alpha = ALPHAS[F % 3]

    def call(c, o, s):
        return lib.a0_loss_quantile(c, 1, qhg.data_ptr(), tng.data_ptr(), thg.data_ptr(), qsg.data_ptr(), F, F, o["grad"],
                                    qbg.data_ptr(), tg.data_ptr(), o["fraction_loss"], o["grad_taus"], s)
    args = (call, B, A, ag, rg, dg, wg, G, alpha, {"grad": (B, F, A), "fraction_loss": (B,), "grad_taus": (B, F + 1)})
    out = launch_twice(*args)
    _set(lib, OPT_QH_SPEC, 0)
    same_bits(f"fqf all-action fetch on/off F={F} A={A}", launch_twice(*args), out)
    _set(lib, OPT_QH_SPEC, 1)
    loss, grad, frac, gt = OL.fqf(qh, taus, th, tn, qb, qs, a, r, d, w, G, 1)
    _, ref64, *_ = _quantile_refs(qh, tn, th, qs, a, r, d, w, G, 1, F, F, True)
    bi = np.arange(B)
    ref64.update(O64.fraction(qh[bi, :, a], qb[bi, :, a], taus, w))
    check(f"shapes.fqf[F={F},A={A}]", out, {"loss": loss, "grad": grad, "fraction_loss": frac, "grad_taus": gt}, ref64, alpha)
