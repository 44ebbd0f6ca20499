"""Device-side timeline of one replay+target step (the -DA0_TRACE build): per kernel launch, when its
CTAs entered, passed griddepcontrol.wait / received their input, and finished (%globaltimer); the edge types of the
captured graph, and for each K4 link which of its predecessors finished last.
Usage: A0_LIB=agent0_b200/libagent0_b200_trace.so python tools/trace_step.py [B] [L] [overlap 0/1]
A0_UNTYPED_JOINS=1,2,4: those links join their wave through the stream wait (programmatic edge) instead of a typed join."""
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("A0_LIB", os.path.join(ROOT, "agent0_b200", "libagent0_b200_trace.so"))
import numpy as np
import torch

import bench as BN
from agent0_b200 import _lib, hotloop
from agent0_b200.config import make_config
from agent0_b200.replay import ReplayDataset

B = int(sys.argv[1]) if len(sys.argv) > 1 else 32
L = int(sys.argv[2]) if len(sys.argv) > 2 else 20
overlap = bool(int(sys.argv[3])) if len(sys.argv) > 3 else True
k4_only = len(sys.argv) > 4 and sys.argv[4] == "k4only"      # the K4 chain alone: are its inputs L2 hits without K3's traffic?
lib = _lib.load()
lib.a0_trace_set.restype = C.c_int
lib.a0_trace_set.argtypes = [C.c_void_p, C.c_void_p]
wl = dict(BN.WORKLOADS["c51_b32"]); wl["B"] = B
cfg = make_config("c51", per=True, n_step=3, batch_size=B, replay_size=1_000_000, double_q=True, dueling=True, num_envs=16, action_dim=4)
rp = ReplayDataset(cfg, native_nstep=True)
BN.fill_shard(rp, 1_000_000, 16, 1234, torch)
BN.GATHER_WINDOW = "auto" if os.environ.get("A0_GATHER_WINDOW", "auto") == "auto" else int(os.environ["A0_GATHER_WINDOW"])
BN.K4_PRIORITY = os.environ.get("A0_K4_PRIORITY", "1") != "0"
_w = os.environ.get("A0_GATHER_WAVES", "auto")             # auto | none | 1,1,2,16 ...: the gather schedule of the step
hp = BN.HotPath(rp, wl, L, 4, torch, waves=_w if _w in ("auto", "none") else [int(x) for x in _w.split(",")])
hp.overlap_sg = overlap
if k4_only:
    hp.rp.push_dynamic()
    hp.step(); hp.step()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        hp.sample()
        for k in range(L):
            hp.target_loss(k)
else:
    if os.environ.get("A0_UNTYPED_JOINS"):
        _untyped = {int(x) for x in os.environ["A0_UNTYPED_JOINS"].split(",")}
        _typed = hotloop.captured_early_links
        hotloop.captured_early_links = lambda L_, w_: _typed(L_, w_) - _untyped
    hp.rp.push_dynamic()
    for _ in range(3):
        hp.step()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph(keep_graph=True)
    with torch.cuda.graph(g):
        hp.step()
    if hp.nodes:
        nE = C.c_int64()
        assert lib.a0_graph_edges(g.raw_cuda_graph(), None, None, None, None, 0, C.byref(nE)) == 0
        cap = nE.value
        ef, et, ety, eport = (C.c_void_p * cap)(), (C.c_void_p * cap)(), (C.c_int32 * cap)(), (C.c_int32 * cap)()
        assert lib.a0_graph_edges(g.raw_cuda_graph(), ef, et, ety, eport, cap, C.byref(nE)) == 0
        E = {(ef[i], et[i]): ("programmatic" if ety[i] else "full") for i in range(nE.value)}
        nd = hp.nodes
        name = {n: f"K4[{k}]" for k, n in enumerate(nd["k4"])}
        name.update({n: f"wave {j}" for j, n in enumerate(nd["waves"])})
        if nd["plan"]:
            name[nd["plan"]] = "plan"
        if nd["apply"]:
            name[nd["apply"]] = "apply"
        print("edges into the K4 links and the apply (captured graph):")
        for n in nd["k4"] + ([nd["apply"]] if nd["apply"] else []):
            print(f"   {name[n]:8s} <- " + ", ".join(f"{name.get(a, 'other')} {t}" for (a, b), t in E.items() if b == n))
    g.instantiate()
for _ in range(5):
    g.replay()
torch.cuda.synchronize()
if os.environ.get("A0_TOUCH_TREE"):            # experiment: pull the whole tree (and the claim scratch) into L2 once
    _ = float(rp.tree.sum())
    for _ in range(int(os.environ["A0_TOUCH_TREE"])):
        g.replay()
    torch.cuda.synchronize()
NREC = 1 << 16
buf = torch.zeros(NREC, 12, dtype=torch.int64, device="cuda")       # {t0, t1, t2, kid | blk << 32, x[4]}
cur = torch.zeros(1, dtype=torch.int32, device="cuda")
assert lib.a0_trace_set(buf.data_ptr(), cur.data_ptr()) == 0
g.replay(); g.replay()
torch.cuda.synchronize()
n = int(cur.item())
rec = buf[:n].cpu().numpy()
lib.a0_trace_set(None, None)
t0, t1, t2 = rec[:, 0], rec[:, 1], rec[:, 2]
kid = (rec[:, 3] & 0xffffffff).astype(np.int64)
# second replay only: split at the largest gap between K2a records
k2 = np.sort(t0[kid == 2])
cut = k2[len(k2) // 2]
sel = t0 >= cut - 500
t0, t1, t2, kid = t0[sel], t1[sel], t2[sel], kid[sel]
xs = rec[sel][:, 4:12]
base = t0.min()
rows = []
names = {2: "K2a", 3: "K3", 4: "K4", 5: "K2b", 7: "K2b plan", 8: "K2b apply"}
if (kid == 4).any():
    t2 = np.where(kid == 4, t0, t2)          # K4's t2 holds cycles, not time
for k in (2, 3, 5, 7, 8):
    m = kid == k
    if m.any():
        rows.append((names[k], int(m.sum()), (t0[m].min() - base) / 1e3, (np.median(t2[m]) - base) / 1e3, (t2[m].max() - base) / 1e3,
                     (t1[m].max() - base) / 1e3))
m = kid == 4
o = np.argsort(t0[m])
per = max(1, int(m.sum()) // L)
for i in range(L):
    s = o[i * per:(i + 1) * per]
    if len(s):
        rows.append((f"K4[{i}]", len(s), (t0[m][s].min() - base) / 1e3, (np.median(t2[m][s]) - base) / 1e3, (t2[m][s].max() - base) / 1e3,
                     (t1[m][s].max() - base) / 1e3))
rows.sort(key=lambda r: r[2])
m4 = kid == 4
if m4.any():
    # K4 stores clock64 (SM cycles) at the wait's return in t2 and at eight points after it
    # x[7] holds the cycle at entry: entry -> wait returned is the batch-side phase plus the wait on an early link
    c0 = rec[sel][:, 2][m4]
    pts = np.concatenate([c0[:, None], xs[m4][:, :7]], 1)
    dd = np.diff(pts, axis=1)
    lab = ["loads land", "arg-max | row maxima", "sum-exps | bin geometry | log-softmax", "p / sum + term weights", "segmented scan + bins",
           "CE | mass reductions", "emit loss / priority / max_p + gradient stores"]
    early = hotloop.captured_early_links(L, hp.waves) if hp.nodes else \
        hotloop.early_links(L, hp.waves, hp._plan_join if hp._use_plan else None)
    t0_4, t1_4 = t0[m4], t1[m4]
    o4 = np.argsort(t0_4)
    per4 = max(1, int(m4.sum()) // L)
    link = np.empty(int(m4.sum()), np.int64)
    for i in range(L):
        link[o4[i * per4:(i + 1) * per4]] = i
    print("K4 (C51) warp-0 phases after griddepcontrol.wait, median SM cycles (1965 cycles = 1 us):")
    for name, ks in (("all links", range(L)), ("early links", sorted(early)), ("join / other links", sorted(set(range(L)) - early))):
        mk = np.isin(link, list(ks))
        if mk.any():
            d = np.median(dd[mk], 0)
            print(f"   {name} ({int(mk.sum())} CTAs): " + " | ".join(f"{l} {int(v)}" for l, v in zip(lab, d)) +
                  f" | total {int(np.median(dd[mk].sum(1)))}")
    # the link-to-link period: last exit of link i-1 -> last exit of link i, by the kind of link i
    ex = np.array([t1_4[link == i].max() for i in range(L)])
    pre = np.array([np.median(c0[link == i] - xs[m4][link == i, 7]) for i in range(L)])
    for name, ks in (("early links", sorted(early)), ("join / other links", sorted(set(range(1, L)) - early))):
        if ks:
            print(f"   {name}: link-to-link period (exit to exit) median {np.median(np.diff(ex)[np.array(ks) - 1]) / 1e3:.2f} us; "
                  f"entry -> wait returned median {int(np.median(pre[ks]))} cycles; links {ks}")
    # which predecessor finished last: the previous link, or the gather wave the link joins (a K3 record carries the
    # first draw of its launch + 1 in x[0])
    wave_exit = {}
    for b0, _, lo, _ in hp.waves or []:
        mw = (kid == 3) & (xs[:, 0] == lo + 1)
        if mw.any():
            wave_exit[b0] = t1[mw].max()
    en = np.array([t0_4[link == i].min() for i in range(L)])
    f_ = lambda v: f"{(v - base) / 1e3:7.2f}" if v is not None else "      -"
    print("   per link, us from the first traced entry: entry | previous link's exit | its wave's exit | exit | link to link"
          " | last predecessor")
    for i in range(L):
        pe, we = (ex[i - 1] if i else None), wave_exit.get(i)
        last = "wave" if we is not None and (pe is None or we > pe) else ("previous link" if pe is not None else "-")
        print(f"   K4[{i:2d}] {'early' if i in early else 'join '} {f_(en[i])} | {f_(pe)} | {f_(we)} | {f_(ex[i])} | "
              f"{(ex[i] - pe) / 1e3 if pe is not None else 0.0:5.2f} | {last}")
m7, m8 = kid == 7, kid == 8
if m7.any() and m8.any() and m4.any():
    print(f"apply: plan exit {(t1[m7].max() - base) / 1e3:.2f} us, last K4 exit {(t1[m4].max() - base) / 1e3:.2f} us: last predecessor "
          f"{'plan' if t1[m7].max() > t1[m4].max() else 'K4[L-1]'}")
m3 = kid == 3
if m3.any():
    q = [0, 10, 50, 90, 100]
    f = lambda a: " ".join("%.2f" % ((np.percentile(a, x) - base) / 1e3) for x in q)
    print("K3 CTAs, percentiles", q, "(us): entry", f(t0[m3]), "| position known", f(t2[m3]), "| exit", f(t1[m3]))
    ent = (t0[m3] - base) / 1e3
    width = max(0.1, float(np.ceil((ent.max() - ent.min()) / 30 * 10) / 10))        # at most ~30 bins
    ent = np.round(np.floor(ent / width) * width, 1)
    vals, cnts = np.unique(ent, return_counts=True)
    print("   entry-time histogram (us: CTAs):", ", ".join(f"{v}: {c}" for v, c in zip(vals, cnts)))
    if os.environ.get("A0_TRACE_LATE"):
        blk = (rec[sel][:, 3] >> 32).astype(np.int64)
        o = np.argsort(-(t2[m3]))[:24]
        k2 = kid == 2
        k2blk = blk[k2]; k2t1 = t1[k2]
        rows_ = []
        for i in o:
            bq = int(blk[m3][i])
            j = np.flatnonzero(k2blk == (bq >> 3))
            rows_.append((bq, round(float(t2[m3][i] - base) / 1e3, 2), round(float(k2t1[j[0]] - base) / 1e3, 2) if len(j) else None))
        print("   latest positions (gather block, known at us, its sampler CTA's warp-0 idx-written at us):", rows_)
    print("   per-CTA gather time (position known -> exit), us: median %.2f  p90 %.2f  max %.2f" % tuple(
        np.percentile((t1[m3] - t2[m3]) / 1e3, [50, 90, 100])))
m5 = kid == 5
if m5.any():
    x5 = xs[m5][0]
    c0 = x5[7]
    lab5 = ["leaves + init", "pass 1 (tickets)", "pass 2 (overlay)", "chunk reduce", "pass 3 (path stores)", "fence + ticket", "roots load"] \
        if os.environ.get("A0_K2B_CHUNKS", "1") != "0" else ["loads + clear + barrier", "insert + ticket", "leaf value", "sparse levels", "heap fill", "dense levels", "write-out"] \
        if os.environ.get("A0_K2B_SMALL", "0") != "0" else \
        ["claim", "leaf write", "release + first climb", "two 3-level climbs", "(to dense)", "dense load", "dense levels"]
    pts = [c0] + [x5[i] for i in range(7)]
    print("K2b (one CTA) phases, SM cycles: " + " | ".join(f"{l} {int(pts[i + 1] - pts[i])}" for i, l in enumerate(lab5)
                                                                 if pts[i + 1] and pts[i]) + f" | total {int(x5[6] - c0)}")
m8 = kid == 8
if m8.any():
    x8 = xs[m8][0]
    lab8 = ["plan + leaves read (before the wait)", "wait", "losses + report + leaves", "climb", "dense top"]
    pts = [x8[7]] + [x8[i] for i in range(5)]
    print("K2b apply, phases of one of its CTAs, SM cycles: " + " | ".join(f"{l} {int(pts[i + 1] - pts[i])}" for i, l in enumerate(lab8))
          + f" | after the wait {int(x8[4] - x8[1])}")
    m4 = kid == 4
    if m4.any():
        print(f"end of the last K4 -> end of the apply: {(t1[m8].max() - t1[m4].max()) / 1e3:.2f} us")
print(f"B={B} L={L} overlap={overlap} gather waves (batches)={[w[1] for w in hp.waves] if hp.waves else None} records={n}; times in us from the first traced entry; globaltimer tick = "
      f"{int(np.min(np.diff(np.unique(np.concatenate([t0, t1])))))} ns")
print(f"{'kernel':8s} {'ctas':>5s} {'first entry':>12s} {'median ready':>13s} {'last ready':>11s} {'last exit':>10s}")
for r in rows:
    print(f"{r[0]:8s} {r[1]:5d} {r[2]:12.2f} {r[3]:13.2f} {r[4]:11.2f} {r[5]:10.2f}")
