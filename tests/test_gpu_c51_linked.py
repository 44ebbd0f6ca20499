"""a0_loss_c51_linked with A0_C51_EARLY: the short-chain C51 kernel reads its batch-side inputs, computes the
projection's geometry and stores the gradient block's zeros before griddepcontrol.wait, and loads only the taken
action's online row after it.  That changes when work is done, never a result: the early kernel is checked against
a0_loss_c51 on the adversarial samples of tests/test_gpu_c51_chain.py, and the batch-32 C51 step of
hotloop.ReplayTargetLoop, graphed and eager, under several gather schedules, with the early links on and off."""
import ctypes as C

import pytest
import torch

from tests.test_gpu_c51_chain import N_CASES, _adversarial
from tests.test_gpu_hotloop import A, _outputs, _shard
from tests.test_gpu_loss_shapes import G3, SUPPORTS, dev, launch, same_bits

pytestmark = pytest.mark.gpu


@pytest.fixture
def lib():
    from agent0_b200 import _lib
    return _lib.load()


@pytest.mark.parametrize("A_", [1, 4, 6])
@pytest.mark.parametrize("M", [2, 33, 51, 64])
def test_early_kernel_matches_the_standalone_call_on_adversarial_samples(lib, M, A_):
    from agent0_b200 import _lib
    B = 2 * N_CASES + 3
    for i, (vmin, vmax) in enumerate(SUPPORTS):
        for G in (G3, 0.0):
            a, r, d, w, atoms, lg, tg, qs = _adversarial(M, A_, B, vmin, vmax, M * 1000 + A_ * 10 + i)
            ag, rg, dg, wg, lgg, tgg, qsg, atg = map(dev, (a, r, d, w, lg, tg, qs, atoms))

            def call(flags):
                if flags is None:
                    return lambda c, o, s: lib.a0_loss_c51(c, lgg.data_ptr(), tgg.data_ptr(), qsg.data_ptr(), atg.data_ptr(),
                                                           M, vmin, vmax, o["grad"], o["target_prob"], s)
                return lambda c, o, s: lib.a0_loss_c51_linked(c, lgg.data_ptr(), tgg.data_ptr(), qsg.data_ptr(),
                                                              atg.data_ptr(), M, vmin, vmax, o["grad"], o["target_prob"],
                                                              flags, s)
            shapes = {"grad": (B, A_, M), "target_prob": (B, M)}
            ref = launch(call(None), B, A_, ag, rg, dg, wg, G, 0.5, shapes)
            for flags in (0, _lib.C51_EARLY):
                same_bits(f"c51 linked flags={flags} M={M} A={A_} ({vmin},{vmax}) G={G}",
                          launch(call(flags), B, A_, ag, rg, dg, wg, G, 0.5, shapes), ref)


def test_linked_rejects_unknown_flags(lib):
    from agent0_b200 import _lib
    c = _lib.LossCommon(B=0, A=4)
    assert lib.a0_loss_c51_linked(C.byref(c), None, None, None, None, 51, -10.0, 10.0, None, None, 2, None) != 0


@pytest.mark.parametrize("waves", ["auto", None, [1] * 20, [2, 2, 4, 12]])
def test_batch32_step_is_the_same_with_and_without_early_links(monkeypatch, waves):
    from agent0_b200 import hotloop
    from agent0_b200.hotloop import ReplayTargetLoop
    Bn, k = 32, 20
    o = _outputs("c51", Bn * k)
    rp_a, rp_b = _shard("c51"), _shard("c51")
    kw = dict(n_step=3, per=True, rng_seed=9, gather_waves=waves, waves_when_eager=True, want_prio=True)
    la, lb = ReplayTargetLoop(rp_a, "c51", Bn, k, A, o, **kw), ReplayTargetLoop(rp_b, "c51", Bn, k, A, o, **kw)
    if waves == "auto":                      # joins: waves at 0, 1, 2, 4, 8 and the plan at 16
        assert len(hotloop.early_links(k, lb.waves, lb._plan_join)) == 14
    elif waves == [2, 2, 4, 12]:             # joins: waves at 0, 2, 4, 8 and the plan at 16
        assert len(hotloop.early_links(k, lb.waves, lb._plan_join)) == 15
    off = lambda *a: frozenset()

    def step_off(fn):
        with monkeypatch.context() as m:
            m.setattr(hotloop, "early_links", off)
            return fn()

    def same():
        torch.cuda.synchronize()
        for f in ("idx", "w", "loss", "newp", "grad"):
            assert torch.equal(getattr(la, f), getattr(lb, f)), f
        assert torch.equal(rp_a.tree, rp_b.tree) and float(rp_a.max_p_tensor) == float(rp_b.max_p_tensor)

    rp_a.push_dynamic(); rp_b.push_dynamic()
    rp_a.rng_seek(0); rp_b.rng_seek(0)
    for _ in range(3):
        lb.grad.fill_(float("nan")); lb.loss.fill_(float("nan"))
        step_off(la.step); lb.step()
        same()
    step_off(lambda: la.capture(warm=1)); lb.capture(warm=1)
    for _ in range(4):
        lb.grad.fill_(float("nan")); lb.loss.fill_(float("nan"))
        la.run(); lb.run()
        same()
