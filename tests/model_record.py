"""What tests/test_model_parity.py compares between agent0_b200.model and the reference's agent0.deepq.model:
one record per network, made by the same code from either package's DeepQNet (tests/golden/make_golden.py
records the reference's side into tests/golden/model_parity.npz)."""
import hashlib

import numpy as np
import torch

ALGOS = ["dqn", "c51", "qr", "iqn", "fqf", "mdqn"]
VARIANTS = [(False, False), (True, False), (True, True)]      # (dueling, noisy)
SAMPLE = 256


def key(algo, dueling, noisy):
    return f"{algo}_{'dueling' if dueling else 'plain'}_{'noisy' if noisy else 'dense'}"


def ortho_names(net):
    """The weights nn.init.orthogonal_ initialises: every Linear / Conv2d except FQF's fraction net (xavier)."""
    return [n + ".weight" for n, m in net.named_modules()
            if isinstance(m, (torch.nn.Linear, torch.nn.Conv2d)) and not n.endswith("fraction_net")]


def record(make_net, algo):
    """``make_net()`` builds the network; the calls run in the order of the original side-by-side comparison:
    seed 3, construct, torch.rand(2), a seeded input, qval under seed 1, forward (IQN / FQF: head(n=8) under
    seed 2, FQF: prop_taus)."""
    torch.manual_seed(3); net = make_net(); r = torch.rand(2)
    sd = net.state_dict()
    ortho = ortho_names(net)
    pick = lambda v, i: np.random.default_rng(i).choice(v.numel(), min(SAMPLE, v.numel()), replace=False)
    out = {"names": np.array(list(sd.keys())),
           "shapes": np.array(["x".join(map(str, v.shape)) for v in sd.values()]),
           "sha256": np.array([hashlib.sha256(v.contiguous().numpy().tobytes()).hexdigest() for v in sd.values()]),
           "ortho": np.array([k in ortho for k in sd]),
           "ortho_sample": np.stack([sd[k].reshape(-1)[pick(sd[k], i)].numpy() for i, k in enumerate(ortho)]),
           "ortho_sumsq": np.array([float(sd[k].double().square().sum()) for k in ortho]),
           "param_names": np.array([n for n, _ in net.named_parameters()]),
           "param_count": np.array(sum(p.numel() for p in net.params())),
           "rand_after_init": r.numpy()}
    x = torch.rand(3, 4, 84, 84)
    torch.manual_seed(1); out["qval"] = net.qval(x).detach().numpy()
    if algo in ("iqn", "fqf"):
        enc = net.encoder(x)
        torch.manual_seed(2); y, t = net.head(enc, n=8)
        out["head_out"], out["head_taus"] = y.detach().numpy(), t.detach().numpy()
    else:
        out["forward"] = net(x).detach().numpy()
    if algo == "fqf":
        for name, v in zip(("taus", "taus_hat", "entropies"), net.head.prop_taus(enc)):
            out["prop_" + name] = v.detach().numpy()
    return out
