"""The short-chain C51 kernel a0_k4_c51_fast against the general a0_k4_c51, on the inputs where their arithmetic could
part ways.

a0_k4_c51_fast computes the bin positions b = (tz - vmin) / delta with a float64 Markstein step from the host's
1/delta instead of an IEEE float32 division (a0_c51_div_delta), and the row maxima with redux.sync.max.f32 instead of an
fmaxf butterfly.  The first test checks the division against __fdiv_rn for every float32 numerator the kernel can see
(every nu in [0, fl32(vmax - vmin)]) on every support and atom count of tests/test_gpu_loss_shapes.py; the second checks
both kernels bit for bit on adversarial samples: exact ties, rows of equal values, +-0 maxima, -inf and NaN entries,
huge offsets, terminal and clamped returns, returns that put tz exactly on vmin, vmax or a bin edge, and NaN selection
values, where both must pick torch.argmax's action (the first NaN) in every lane, as oracle/losses64.py does."""
import numpy as np
import pytest
import torch

from oracle import losses64 as O64
from tests.test_gpu_loss_shapes import G3, OPT_C51_FAST, SUPPORTS, bound64, dev, launch, nan_selection_rows, same_bits

pytestmark = pytest.mark.gpu

f32 = np.float32
MS = [2, 3, 31, 32, 33, 63, 64]          # the atom counts of test_c51_fast_eligible_shapes


@pytest.fixture
def lib():
    from agent0_b200 import _lib
    L = _lib.load()
    yield L
    L.a0_set_option(OPT_C51_FAST, 1)


@pytest.mark.parametrize("vmin,vmax", SUPPORTS)
def test_bin_division_is_correctly_rounded_for_every_numerator(lib, vmin, vmax):
    from agent0_b200 import _lib
    hi = f32(f32(vmax) - f32(vmin))
    n = int(np.array(hi).view(np.uint32)) + 1
    for M in MS:
        out = torch.tensor([0, -1], dtype=torch.int64, device="cuda")      # mismatches, first mismatching bit pattern
        _lib.check(lib.a0_c51_div_check(vmin, vmax, M, out.data_ptr(), _lib.stream_ptr()), "a0_c51_div_check")
        bad, first = out.cpu().tolist()
        assert bad == 0, (f"({vmin}, {vmax}), M = {M}: {bad} of {n} numerators differ from __fdiv_rn, the first "
                          f"{np.array(first & 0xffffffff, np.uint32).view(f32)!r}")


N_CASES = 27
SEL_CASES = 21                         # cases SEL_CASES.. are NaN selection values (nan_selection_rows)


def _adversarial(M, A, B, vmin, vmax, seed):
    """Sample b is special case b % N_CASES on top of random rows."""
    rng = np.random.RandomState(seed)
    atoms = np.linspace(vmin, vmax, M).astype(f32)
    delta = f32(f32(f32(vmax) - f32(vmin)) / f32(M - 1))
    a = rng.randint(0, A, B).astype(np.int64)
    r = rng.choice([-1.0, 0.0, 1.0, 0.4], B).astype(f32)
    d = (rng.rand(B) < 0.25).astype(f32)
    w = (rng.rand(B) + 0.05).astype(f32)
    lg, tg = [(rng.randn(B, A, M) * 3).astype(f32) for _ in range(2)]
    qs = (rng.randn(B, A) * 3).astype(f32)
    k = M // 2
    for b in range(B):
        c = b % N_CASES
        if c == 0:                                     # rows of equal values
            lg[b], tg[b] = 1.5, -2.0
        elif c == 1:                                   # +0 and -0 tie for the maximum
            lg[b] = -np.abs(lg[b]); lg[b, :, ::2] = 0.0; lg[b, :, 1::2] = -0.0
            tg[b] = -np.abs(tg[b]); tg[b, :, ::3] = -0.0; tg[b, :, 1::3] = 0.0
        elif c in (2, 3):                              # a lone -0 / +0 maximum: exp(-200) is 0, so lse = 0, and all mass
            j = k if c == 2 else 0                     # on one bin
            lg[b] = -200.0; lg[b, :, j] = -0.0 if c == 2 else 0.0
            r[b], d[b] = atoms[j], 1.0
        elif c == 4:                                   # -inf entries
            lg[b, :, ::3] = -np.inf; tg[b, :, 1::2] = -np.inf
        elif c == 5:                                   # one finite target logit
            tg[b] = -np.inf; tg[b, :, M - 1] = 4.0
        elif c == 6:                                   # huge offsets
            lg[b] += f32(1e30); tg[b] += f32(1e6)
        elif c == 7:                                   # the largest finite logits
            lg[b, :, 0] = f32(3.4e38); tg[b, :, M - 1] = f32(-3.4e38)
        elif c == 8:                                   # NaN in the online row
            lg[b, :, M // 3] = np.nan
        elif c == 9:                                   # NaN in the target row
            tg[b, :, M - 1] = np.nan
        elif c == 10:                                  # an online row of -inf
            lg[b] = -np.inf
        elif c == 11:                                  # tied selection values: the first wins
            qs[b] = 0.5
        elif c == 12:                                  # tz on vmin, on vmax, on bin edges, just above an atom
            r[b], d[b] = vmin, 1.0
        elif c == 13:
            r[b], d[b] = vmax, 1.0
        elif c == 14:
            r[b], d[b] = f32(f32(vmin) + f32(k * delta)), 1.0
        elif c == 15:
            r[b], d[b] = atoms[min(1, M - 1)], 1.0
        elif c == 16:
            r[b], d[b] = np.nextafter(atoms[k], f32(np.inf)), 1.0
        elif c == 17:                                  # every atom clamped at vmax
            r[b] = 1000.0
        elif c == 18:                                  # ... at vmin
            r[b] = -1000.0
        elif c == 19:                                  # shifted by whole bins (with gamma_n = 1: tz = z + 3 delta)
            r[b], d[b] = f32(3 * delta), 0.0
        elif c >= SEL_CASES:                           # random rows, NaN selection values
            qs[b] = nan_selection_rows(A)[c - SEL_CASES]
        else:
            r[b], d[b] = 0.0, 0.0
    return a, r, d, w, atoms, lg, tg, qs


@pytest.mark.parametrize("A", [1, 4, 6])
@pytest.mark.parametrize("M", [2, 3, 33, 51, 64])
def test_fast_kernel_matches_general_on_adversarial_samples(lib, M, A):
    B = 2 * N_CASES + 3                                # every case at least twice, a partial last CTA
    for i, (vmin, vmax) in enumerate(SUPPORTS):
        for G in (G3, 1.0, 0.0):
            a, r, d, w, atoms, lg, tg, qs = _adversarial(M, A, B, vmin, vmax, M * 1000 + A * 10 + i)
            ag, rg, dg, wg, lgg, tgg, qsg, atg = map(dev, (a, r, d, w, lg, tg, qs, atoms))

            def call(c, o, s):
                return lib.a0_loss_c51(c, lgg.data_ptr(), tgg.data_ptr(), qsg.data_ptr(), atg.data_ptr(), M, vmin, vmax,
                                       o["grad"], o["target_prob"], s)
            args = (call, B, A, ag, rg, dg, wg, G, 0.5, {"grad": (B, A, M), "target_prob": (B, M)})
            assert lib.a0_set_option(OPT_C51_FAST, 0) == 0
            general = launch(*args)
            assert lib.a0_set_option(OPT_C51_FAST, 1) == 0
            fast = launch(*args)
            same_bits(f"c51 fast vs general, adversarial M={M} A={A} ({vmin},{vmax}) G={G}", fast, general)
            same_bits(f"c51 fast, second launch M={M} A={A}", launch(*args), fast)
            sel = np.arange(B) % N_CASES >= SEL_CASES
            ref64 = O64.c51(lg[sel], tg[sel], qs[sel], a[sel], r[sel], d[sel], w[sel], G, atoms, vmin, vmax)
            for k in ("loss", "target_prob", "grad"):
                bound64(f"c51 NaN selection M={M} A={A} ({vmin},{vmax}) G={G}.{k}", fast[k][sel], ref64[k])
