"""The captured waved step read back from its CUDA graph (a0_graph_edges on raw_cuda_graph()): the K4 links are chained by
programmatic edges, the links of ``captured_early_links`` take their gather wave through a full (default-typed) edge, the
write-back plan joins the apply through a full edge and no K4 link, and the step computes what it computes issued eagerly."""
import ctypes as C

import pytest
import torch

from agent0_b200 import _lib
from agent0_b200.hotloop import ReplayTargetLoop, captured_early_links
from tests.test_gpu_hotloop import _outputs, _shard

pytestmark = pytest.mark.gpu
DEFAULT, PROGRAMMATIC = 0, 1            # cudaGraphDependencyType


def _edges(graph):
    """{(from, to): edge type} of a cudaGraph_t."""
    lib, n = _lib.load(), C.c_int64()
    _lib.check(lib.a0_graph_edges(graph, None, None, None, None, 0, C.byref(n)), "a0_graph_edges")
    cap = n.value
    f, t, ty, port = (C.c_void_p * cap)(), (C.c_void_p * cap)(), (C.c_int32 * cap)(), (C.c_int32 * cap)()
    _lib.check(lib.a0_graph_edges(graph, f, t, ty, port, cap, C.byref(n)), "a0_graph_edges")
    return {(f[i], t[i]): ty[i] for i in range(n.value)}


def _loop(algo, Bn, L, eager=False):
    rp = _shard(algo)
    lp = ReplayTargetLoop(rp, algo, Bn, L, 4, _outputs(algo, Bn * L), n_step=3, rng_seed=11, waves_when_eager=eager)
    rp.push_dynamic()
    return rp, lp


@pytest.mark.parametrize("algo,Bn,L", [("c51", 32, 20), ("dqn", 32, 20), ("c51", 512, 4)])
def test_captured_step_edges(algo, Bn, L):
    rp, lp = _loop(algo, Bn, L)
    lp.step()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph(keep_graph=True)
    with torch.cuda.graph(g):
        lp.step()
    E, nd = _edges(g.raw_cuda_graph()), lp.nodes
    k4, waves = nd["k4"], nd["waves"]
    assert len(k4) == L and len(waves) == len(lp.waves)
    for k in range(1, L):
        assert E[(k4[k - 1], k4[k])] == PROGRAMMATIC, k
    typed = captured_early_links(L, lp.waves) if algo == "c51" else frozenset()
    for j, (b0, _, _, _) in enumerate(lp.waves):
        # a typed join takes its wave through a full edge; the others keep the stream wait's programmatic edge
        assert E[(waves[j], k4[b0])] == (DEFAULT if b0 in typed else PROGRAMMATIC), (j, b0)
        assert all(E.get((waves[j], k4[k])) is None for k in range(L) if k != b0)
    if Bn == 32:
        assert typed == (frozenset(range(1, L)) if algo == "c51" else frozenset())
        assert nd["plan"] is not None and nd["apply"] is not None
        assert E[(k4[-1], nd["apply"])] == PROGRAMMATIC
        assert E[(nd["plan"], nd["apply"])] == DEFAULT
        assert all((nd["plan"], n) not in E for n in k4), "a K4 link still joins the write-back plan"
    else:
        assert typed == frozenset() and nd["plan"] is None

    # the captured step computes what the eager one computes on a twin shard, replay after replay
    rq, lq = _loop(algo, Bn, L, eager=True)
    lq.step(); lq.step()                 # the captured loop's warm-up step and first replay
    g.replay()
    for _ in range(3):
        rp.push_dynamic(); g.replay()
        rq.push_dynamic(); lq.step()
        torch.cuda.synchronize()
        for f in ("idx", "w", "act", "r32", "loss", "grad"):
            assert torch.equal(getattr(lp, f), getattr(lq, f)), f
        assert torch.equal(rp.tree.view(torch.int32), rq.tree.view(torch.int32))
