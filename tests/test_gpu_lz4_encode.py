"""K7 (a0_lz4_encode): the device LZ4 encoder produces exactly the bytes of oracle/lz4_encode.py's encode_greedy for
frame sizes 16, 7056 (84x84) and 9216 (96x96, groups above 64 KB) and noise / constant / Atari-like / mixed groups;
K6a (a0_ex_decode) gives the input back; two launches give the same bytes and frame hashes."""
import numpy as np
import pytest
import torch

from agent0_b200 import _lib
from oracle.lz4_encode import encode_greedy
from tests.test_lz4_encode_oracle import synth_groups

pytestmark = pytest.mark.gpu
HW = {16: (4, 4), 7056: (84, 84), 9216: (96, 96)}


def _groups(F, kind, count, seed, hw=None):
    rng = np.random.RandomState(seed)
    if kind == "noise":
        return [rng.randint(0, 256, 8 * F, dtype=np.uint8).tobytes() for _ in range(count)]
    if kind == "constant":
        return [bytes([int(rng.randint(0, 256))]) * (8 * F) for _ in range(count)]
    syn = synth_groups(count, seed=seed, hw=hw or HW[F])
    if kind == "synthetic":
        return syn
    out = []                                   # mixed: frames of a group alternate between Atari-like and noise
    for g in syn:
        a = np.frombuffer(g, np.uint8).reshape(8, F).copy()
        a[1::2] = rng.randint(0, 256, (4, F), dtype=np.uint8)
        out.append(a.tobytes())
    return out


def encode(groups, F):
    lib = _lib.load()
    m = len(groups)
    frames = torch.tensor(np.frombuffer(b"".join(groups), np.uint8).copy(), device="cuda")
    stride = _lib.lz4_stride(F)
    out = torch.zeros(m * stride, dtype=torch.uint8, device="cuda")
    ln = torch.zeros(m, dtype=torch.int32, device="cuda")
    hs = torch.zeros(m * 8, dtype=torch.int64, device="cuda")
    _lib.check(lib.a0_lz4_encode(frames.data_ptr(), m, F, out.data_ptr(), ln.data_ptr(), hs.data_ptr(), _lib.stream_ptr()),
               "a0_lz4_encode")
    torch.cuda.synchronize()
    o, n = out.cpu().numpy(), ln.cpu().numpy()
    return [o[i * stride:i * stride + int(n[i])].tobytes() for i in range(m)], hs.cpu()


def _shard(F):
    from agent0_b200.config import make_config
    from agent0_b200.replay import ReplayDataset
    cfg = make_config("dqn", replay_size=64, num_envs=2)
    cfg.obs_shape = (4,) + HW[F]
    return ReplayDataset(cfg)


@pytest.mark.parametrize("F", [16, 7056, 9216])
@pytest.mark.parametrize("kind", ["noise", "constant", "synthetic", "mixed"])
def test_k7_equals_encode_greedy_and_decodes(F, kind):
    groups = _groups(F, kind, 5, seed=F + len(kind))
    blobs, hashes = encode(groups, F)
    for g, b in zip(groups, blobs):
        assert b == encode_greedy(g)
    if kind == "noise" and F > 16:
        assert all(len(b) == 8 * F for b in blobs)                   # stored raw
    if kind == "constant" and F > 16:
        assert all(len(b) < 8 * F // 50 for b in blobs)
    rp = _shard(F)
    dec, status = rp.decode_entries(blobs)
    assert (status == 0).all()
    assert dec.cpu().numpy().tobytes() == b"".join(groups)
    blobs2, hashes2 = encode(groups, F)
    assert blobs2 == blobs and torch.equal(hashes, hashes2)
    h = hashes.view(-1, 8)
    flat = np.frombuffer(b"".join(groups), np.uint8).reshape(-1, F)
    for i in range(flat.shape[0]):                                  # equal frames <=> equal hashes (on these inputs)
        for j in range(i):
            assert (int(h.view(-1)[i]) == int(h.view(-1)[j])) == bool((flat[i] == flat[j]).all())
