"""Time of the neighbourhood link-prediction heuristics (ops.simple_adjacency, ops.link_heuristics) and the fb-pages-food table.
  adjacency build     R-MAT 1M nodes / 16M edge samples, the test split's message-passing graph (train + val edges)
  link_heuristics     that split's test pairs (~3 M), a collab-scale ranking table (R-MAT 2^18 / 1.3 M: 50 000 x 101 pairs) and
                      a stress case, 10^4 pairs among the 64 highest-degree nodes of the R-MAT graph
each against a plain torch formulation of the same scores, alternating in one process: the shorter list of each pair expanded
with repeat_interleave, torch.searchsorted over the sorted (row, neighbour) keys, index_add_ segment sums. cn and jaccard must
be equal, aa and ra within 0.5 ulp32 + 2 c 2^-53 of the torch float64 sums. CUDA-event time, median of `reps` after one warm-up; the
times include the op's one host read. Probes = sum over the pairs of min(d(u), d(v)).
Then AUC, hits@20/50/100 (test split, shared negatives) and MRR (100 filtered negatives per positive) of each heuristic on the
fb-pages-food seed-0 split (tests/golden/fb_pages_food_seed0.npz).      python tools/bench_heuristics.py [reps]"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "link-prediction-gnn_b200")):
    sys.path.insert(0, p)
import numpy as np
import torch

import bench
import TwoWL.operators.datasets as D
from TwoWL.model.train import heuristic_scores, rank_scores
from TwoWL.operators.synthetic import rmat_edges
from twowl_b200 import ops

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 9
dev = torch.device("cuda", 0)
try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True, timeout=60).stdout.strip()
except (OSError, subprocess.SubprocessError):
    card = ""
print(f"# card: {card or torch.cuda.get_device_name(dev) + ' (power limit not read)'}", flush=True)


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), out


def timed(fn):
    fn()
    ts = []
    for _ in range(reps):
        t, out = event_ms(fn)
        ts.append(t)
    return sorted(ts)[reps // 2], out


def duel(ours, theirs):
    """alternate the two, `reps` times each after one warm-up of both -> (our ms, their ms, our result, their result)."""
    r0, r1 = ours(), theirs()
    t0, t1 = [], []
    for _ in range(reps):
        t, r0 = event_ms(ours)
        t0.append(t)
        t, r1 = event_ms(theirs)
        t1.append(t)
    return sorted(t0)[reps // 2], sorted(t1)[reps // 2], r0, r1


def split_graph(workload, seed=0):
    scale, samples, abcd, _ = bench.WORKLOADS[workload]
    s, d, _ = rmat_edges(scale, samples, abcd, seed, dev)
    bg = D.graph_from_split(D.do_edge_split(D._Data(torch.stack((s, d)))), pattern="none")   # no wedge index: no model here
    bg.preprocess()
    bg.setPosDegreeFeature()
    return bg


def torch_heuristics(keys, ptr, adj, u, v):
    """The same scores in plain torch -> (fp32 [4, P], aa float64, ra float64)."""
    n, P = ptr.numel() - 1, u.numel()
    deg = ptr.diff()
    du, dv = deg[u], deg[v]
    swap = (du > dv) | ((du == dv) & (u > v))
    s, l = torch.where(swap, v, u), torch.where(swap, u, v)
    ds = deg[s]
    pair = torch.repeat_interleave(torch.arange(P, device=dev), ds)
    first = torch.cumsum(ds, 0) - ds
    x = adj[ptr[s][pair] + torch.arange(pair.numel(), device=dev) - first[pair]].long()
    q = l[pair] * n + x
    pos = torch.searchsorted(keys, q).clamp_(max=max(keys.numel() - 1, 0))
    hit = keys[pos] == q
    p, w = pair[hit], x[hit]
    dw = deg[w].double()
    cn = torch.zeros(P, dtype=torch.int64, device=dev).index_add_(0, p, torch.ones_like(p))
    aa = torch.zeros(P, dtype=torch.float64, device=dev).index_add_(0, p, torch.where(dw > 1, 1.0 / dw.clamp(min=2).log(), 0.0))
    ra = torch.zeros(P, dtype=torch.float64, device=dev).index_add_(0, p, 1.0 / dw)
    den = du + dv - cn
    jac = torch.where(den > 0, cn.float() / den.float().clamp(min=1), torch.zeros((), device=dev))
    return torch.stack((cn.float(), jac, aa.float(), ra.float())), aa, ra


def compare(a, b, name):
    """ours (fp32) against the torch formulation (cn / jaccard fp32, aa / ra float64)"""
    assert torch.equal(a[:2], b[0][:2]), f"{name}: cn / jaccard differ"
    c = a[0].double()
    for r, ref in ((2, b[1]), (3, b[2])):
        r32 = ref.abs().float()
        ulp = (torch.nextafter(r32, torch.full_like(r32, float("inf"))) - r32).double()
        err = (a[r].double() - ref).abs()
        assert bool((err <= 0.5 * ulp + 2 * c * 2.0 ** -53 * ref.abs()).all()), f"{name}: {ops.HEURISTICS[r]} off by {float(err.max())}"


def case(name, ptr, adj, keys, u, v):
    deg = ptr.diff()
    probes = int(torch.minimum(deg[u], deg[v]).sum())
    m0, m1, a, b = duel(lambda: ops.link_heuristics(ptr, adj, u, v), lambda: torch_heuristics(keys, ptr, adj, u, v))
    compare(a, b, name)
    print(f"{name:44s} P={u.numel():9d}  probes={probes:12d}  ours {m0:9.3f} ms ({probes / m0 / 1e6:7.2f} G probes/s)   "
          f"torch {m1:9.3f} ms   x{m1 / m0:.1f}", flush=True)


def row_keys(ptr, adj):
    n = ptr.numel() - 1
    return torch.repeat_interleave(torch.arange(n, device=dev), ptr.diff()) * n + adj.long()


# ---- R-MAT 1M / 16M: adjacency build, the test split, the hub stress case
bg = split_graph("rmat")
tst = D.dataset(*bg.split(2))
n, ei = bg.num_nodes, tst.ei
ms, (ptr, adj) = timed(lambda: ops.simple_adjacency(ei[0], ei[1], n))
deg = ptr.diff()
print(f"{'simple_adjacency  R-MAT 1M/16M':44s} E={ei.shape[1]:9d}  nnz={adj.numel():11d}  max deg={int(deg.max())}  "
      f"ours {ms:9.3f} ms (incl. the host read of nnz)", flush=True)
keys = row_keys(ptr, adj)
E = ei.shape[1]
pairs = tst.pos1[E::2]
case("link_heuristics  R-MAT test split", ptr, adj, keys, pairs[:, 0].contiguous(), pairs[:, 1].contiguous())
g = torch.Generator(device=dev).manual_seed(0)
hubs = torch.topk(deg, 64).indices
hu, hv = hubs[torch.randint(0, 64, (10_000,), generator=g, device=dev)], hubs[torch.randint(0, 64, (10_000,), generator=g, device=dev)]
case("link_heuristics  10^4 pairs among top-64 hubs", ptr, adj, keys, hu, hv)
del bg, tst, ptr, adj, keys, pairs
torch.cuda.empty_cache()

# ---- collab scale: a ranking table of 50 000 positives x (1 + 100) pairs
bg = split_graph("collab")
rk = D.ranking_dataset(bg, 2, num_neg=100)
n, E = bg.num_nodes, rk.ei.shape[1]
ptr, adj = ops.simple_adjacency(rk.ei[0], rk.ei[1], n)
und = rk.pos1[E::2]
Pp = und.shape[0] // 101
und = torch.cat((und[:50_000], und[Pp:].reshape(Pp, 100, 2)[:50_000].reshape(-1, 2)))
case("link_heuristics  collab table 50000 x 101", ptr, adj, row_keys(ptr, adj), und[:, 0].contiguous(), und[:, 1].contiguous())
del bg, rk, ptr, adj
torch.cuda.empty_cache()

# ---- fb-pages-food seed-0: the heuristics next to the reference's recorded baselines (BASELINE.md)
fb = np.load(os.path.join(ROOT, "tests", "golden", "fb_pages_food_seed0.npz"))
nf = int(fb["num_nodes"][0])
ep, en = (torch.from_numpy(fb[k].astype(np.int64)).to(dev) for k in ("edge_pos", "edge_neg"))
bg = D.BaseGraph(torch.zeros((nf, 0), device=dev), None, ep, en, torch.from_numpy(fb["num_pos"]), torch.from_numpy(fb["num_neg"]),
                 "none")
bg.preprocess()
bg.setPosDegreeFeature()
tst = D.dataset(*bg.split(2))
rk = D.ranking_dataset(bg, 2, num_neg=100)
h, hr = heuristic_scores(tst), heuristic_scores(rk)
labels = tst.y.reshape(-1)[0::2]
print(f"# fb-pages-food seed 0, test split: {labels.numel()} pairs ({int(labels.sum())} positives); MRR over 100 filtered negatives")
print(f"{'heuristic':10s} {'AUC':>8s} {'hits@20':>8s} {'hits@50':>8s} {'hits@100':>8s} {'MRR':>8s}")
for name in ops.HEURISTICS:
    auc = float(ops.auc(h[name], labels)[0])
    hk = rank_scores(h[name], tst, (20, 50, 100))
    mrr = rank_scores(hr[name], rk, (20,))["mrr"]
    print(f"{name:10s} {auc:8.4f} {hk['hits@20']:8.4f} {hk['hits@50']:8.4f} {hk['hits@100']:8.4f} {mrr:8.4f}", flush=True)
