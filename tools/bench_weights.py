"""Weight snapshots for actors (K8, agent0_b200/weights.py) against what they replace, on the C51 dueling Nature-CNN
state (1 814 994 fp32 words, 7.26 MB: the flat buffer broadcast_model sends).

  publish            WeightPublisher.publish, CUDA events around each of --iters launches
  fetch_same_gpu     WeightSubscriber fetch (fetch + apply kernels) of a new version on the same GPU, in-process
                     attach; events around the fetch only, a publish before each
  fetch_peer_gpu     (two GPUs) a subscriber process on cuda:1 mapping the handle of cuda:0 over NVLink, while this
                     process keeps publishing: events around each fetch that applied a version
  state_dict_host    state_dict() -> .cpu() -> load_state_dict on the actor's GPU (launch.py:33-36 without the pickling
                     and the RPC), host clock around synchronised iterations
  broadcast_model    actor.broadcast_model over NCCL in a world of one (pack, collective, unpack; no second rank)

Achieved bandwidth counts 2 x 7.3 MB per publish (read the tensors, write the buffer) and per fetch stage.  One JSON
object (card name, power limit and clocks read in the same run) to stdout, and to --out."""
import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from agent0_b200.config import make_config  # noqa: E402
from agent0_b200.model import DeepQNet  # noqa: E402
from agent0_b200.weights import WeightPublisher, WeightSubscriber  # noqa: E402


def _cfg():
    return make_config("c51", per=True, n_step=3, batch_size=32, double_q=True, dueling=True)


def _net(device, seed):
    torch.manual_seed(seed)
    return DeepQNet(_cfg()).to(device)


def _events(n):
    return [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]


def _stats(us):
    us = np.asarray(us, dtype=np.float64)
    return dict(mean_us=float(us.mean()), median_us=float(np.median(us)), p10_us=float(np.percentile(us, 10)),
                p90_us=float(np.percentile(us, 90)), n=int(us.size))


def _peer_child(handle, iters, ready, results):
    out = dict(error=None, us=[])
    try:
        torch.cuda.set_device(1)
        actor = _net("cuda:1", 2)
        sub = WeightSubscriber(handle, actor)
        ready.set()
        ev = _events(iters)
        sts = torch.zeros(iters, dtype=torch.int64, device="cuda:1")
        deadline = time.monotonic() + 60
        for i, (a, b) in enumerate(ev):
            if time.monotonic() > deadline:
                break
            a.record()
            st = sub.pull_async()
            b.record()
            sts[i:i + 1].copy_(st)
            time.sleep(200e-6)
        torch.cuda.synchronize()
        s = sts.cpu().numpy()
        out["us"] = [a.elapsed_time(b) * 1e3 for (a, b), v in zip(ev, s) if v]
        out["pulls"] = int(len(s))
        sub.close()
    except Exception as e:
        out["error"] = repr(e)
    finally:
        ready.set()
        results.put(out, timeout=10)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=500)
    ap.add_argument("--out")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_weights needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    learner, actor = _net(dev, 1), _net(dev, 2)
    pub = WeightPublisher(learner)
    sub = WeightSubscriber(pub, actor)
    n_bytes = pub.n_words * 4
    res = dict(tool="bench_weights", gpus=smi, state="c51 dueling Nature-CNN", n_words=pub.n_words, bytes=n_bytes,
               iters=a.iters)
    for _ in range(20):                                           # warm-up
        pub.publish()
        sub.pull()

    ev = _events(a.iters)
    for e0, e1 in ev:
        e0.record()
        pub.publish()
        e1.record()
    torch.cuda.synchronize()
    res["publish"] = _stats([e0.elapsed_time(e1) * 1e3 for e0, e1 in ev])

    ev = _events(a.iters)
    st = None
    for e0, e1 in ev:
        pub.publish()
        e0.record()
        st = sub.pull_async()
        e1.record()
    torch.cuda.synchronize()
    assert int(st[0]) > 0
    res["fetch_same_gpu"] = _stats([e0.elapsed_time(e1) * 1e3 for e0, e1 in ev])
    for k in ("publish", "fetch_same_gpu"):
        res[k]["achieved_TBps"] = 2 * n_bytes / (res[k]["median_us"] * 1e-6) / 1e12
    res["fetch_same_gpu"]["note"] = "fetch kernel (region -> staging) + apply kernel (staging -> tensors)"

    host = []
    for _ in range(min(a.iters, 100)):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sd = {k: v.cpu() for k, v in learner.state_dict().items()}
        actor.load_state_dict(sd)
        torch.cuda.synchronize()
        host.append((time.perf_counter() - t0) * 1e6)
    res["state_dict_host"] = _stats(host[5:])

    import torch.distributed as dist
    from agent0_b200.actor import broadcast_model
    with tempfile.TemporaryDirectory() as d:
        dist.init_process_group("nccl", store=dist.FileStore(os.path.join(d, "store"), 1), rank=0, world_size=1,
                                device_id=dev)
        try:
            bc = []
            for i in range(min(a.iters, 200) + 10):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                broadcast_model(learner, src=0)
                torch.cuda.synchronize()
                bc.append((time.perf_counter() - t0) * 1e6)
            res["broadcast_model_world1"] = _stats(bc[10:])
        finally:
            dist.destroy_process_group()

    if torch.cuda.device_count() >= 2:
        ctx = mp.get_context("spawn")
        results, ready = ctx.Queue(), ctx.Event()
        p = ctx.Process(target=_peer_child, args=(pub.handle(), a.iters, ready, results), daemon=True)
        p.start()
        try:
            ready.wait(timeout=120)
            t_end = time.monotonic() + 90
            out = None
            while out is None and time.monotonic() < t_end:
                pub.publish()
                torch.cuda.synchronize()
                time.sleep(100e-6)
                try:
                    out = results.get_nowait()
                except Exception:
                    pass
            p.join(timeout=30)
        finally:
            if p.is_alive():
                p.terminate()
                p.join(timeout=10)
        if out and not out["error"] and out["us"]:
            res["fetch_peer_gpu"] = _stats(out["us"])
            res["fetch_peer_gpu"]["pulls"] = out["pulls"]
            res["fetch_peer_gpu"]["note"] = "subscriber process on cuda:1, publisher on cuda:0 publishing concurrently"
        else:
            res["fetch_peer_gpu"] = dict(error=(out or {}).get("error", "no result"))
    else:
        res["fetch_peer_gpu"] = "not measured: one GPU"
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
