"""agent0_b200.model against the reference's agent0.deepq.model on CPU: same seed -> the same state_dict
(names, shapes, values), same RNG consumption, same outputs.

Both tests compare with outputs of the reference's own DeepQNet:
  * tests/golden/act.npz (make_golden.py gen_act): the q-values the unmodified Actor.act computed with the
    DeepQNet it built after torch.manual_seed(7) -- a plain DQN and a dueling C51 network, six calls each;
  * tests/golden/model_parity.npz (make_golden.py gen_model_parity): per network of the six algorithms x
    {plain, dueling, dueling + noisy}, the record of tests/model_record.py.  make_golden.py can only write it
    where the reference package is importable; until it has been recorded that test skips.

Bits that depend on the host are compared with a bound: orthogonal_ initialises through a QR factorisation
whose rounding depends on the LAPACK build and its thread count, so for each of those weights a seeded
sample of 256 values agrees to 1e-5 of the sample's largest magnitude and the sum of squares to 1e-5
relative (measured: 2e-6 between 1, 2, 3 and 8 threads), and the network outputs computed from them to 1e-4 of the output's largest magnitude
(measured: 1.1e-5, C51's qval sums atoms of +-10 with cancellation).  Every other tensor, and the RNG draw,
must be bit-identical."""
import os

import numpy as np
import pytest
import torch

from tests.model_record import ALGOS, VARIANTS, key, record

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden", "model_parity.npz")
W_TOL, OUT_TOL = 1e-5, 1e-4


def _close(got, want, tol):
    return got.shape == want.shape and np.abs(got - want).max() <= tol * np.abs(want).max()


@pytest.mark.parametrize("algo", ["dqn", "c51"])
def test_seeded_network_computes_the_reference_actors_q_values(golden, algo):
    """gen_act: torch.manual_seed(7), then the reference Actor built DeepQNet (action_dim 4, dueling for C51)
    and Actor.act evaluated qval on obs / 255 of the recorded stream, six times."""
    from agent0_b200.config import make_config
    from agent0_b200.model import DeepQNet
    from agent0_b200.synth import record_stream
    g = golden("act")
    s = record_stream(16, 6, seed=321, p_terminal=0.05, p_life_loss=0.05, p_truncated=0.02)
    assert np.array_equal(s["obs"][0], g[f"{algo}_obs_first"])
    torch.manual_seed(7)
    net = DeepQNet(make_config(algo, dueling=(algo == "c51"), action_dim=4))
    with torch.no_grad():
        for k in range(len(g["epsilon"])):
            q = net.qval(torch.from_numpy(s["obs"][k]).float() / 255).numpy()
            assert _close(q, g[f"{algo}_q"][k], OUT_TOL), k


@pytest.mark.skipif(not os.path.exists(GOLDEN), reason="tests/golden/model_parity.npz not recorded yet "
                                                       "(make_golden.py gen_model_parity, from the reference package)")
@pytest.mark.parametrize("algo", ALGOS)
@pytest.mark.parametrize("dueling,noisy", VARIANTS)
def test_same_seed_same_network(algo, dueling, noisy):
    from agent0_b200.config import make_config
    from agent0_b200.model import DeepQNet
    with np.load(GOLDEN, allow_pickle=False) as g:
        want = {k.split("/", 1)[1]: g[k] for k in g.files if k.startswith(key(algo, dueling, noisy) + "/")}
    got = record(lambda: DeepQNet(make_config(algo, dueling=dueling, noisy_net=noisy, action_dim=6)), algo)
    assert sorted(got) == sorted(want)
    assert list(got["names"]) == list(want["names"])
    assert list(got["shapes"]) == list(want["shapes"])
    assert np.array_equal(got["ortho"], want["ortho"])
    for name, a, b, qr in zip(got["names"], got["sha256"], want["sha256"], want["ortho"]):
        assert qr or a == b, f"{name}: values differ from the reference's"
    assert np.array_equal(got["rand_after_init"], want["rand_after_init"])    # constructors consumed the RNG identically
    assert list(got["param_names"]) == list(want["param_names"])
    assert int(got["param_count"]) == int(want["param_count"])
    for i, (a, b) in enumerate(zip(got["ortho_sample"], want["ortho_sample"])):   # one row per orthogonal weight
        assert _close(a, b, W_TOL), f"orthogonal weight {i}"
    assert np.all(np.abs(got["ortho_sumsq"] - want["ortho_sumsq"]) <= W_TOL * np.abs(want["ortho_sumsq"]))
    for k in got:
        if got[k].dtype.kind == "f" and not k.startswith("ortho") and k != "rand_after_init":
            assert _close(got[k], want[k], OUT_TOL), k
