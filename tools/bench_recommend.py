"""Time of link recommendation (ops.recommend_links) and its recall on fb-pages-food.
  R-MAT 1M nodes / 16M edge samples, the test split's message-passing graph (train + val edges):
    the sources of the first 10^4 test positives, k = 100, for each heuristic, and the max-degree node alone;
  each against a plain torch formulation of the same op, alternating in one process: the two-hop expansion with
  repeat_interleave, torch.unique over (query, v) keys, index_add_ sums, then the per-query order by two
  stable sorts, in batches of the same expansion budget. ids must be equal for cn / jaccard; for aa and ra they may differ only
  where adjacent candidates' scores lie within 0.5 ulp32 + 2 c 2^-53, because index_add_ adds the terms in another order (the
  tests check ra bit for bit against a sequential restatement).
  CUDA-event time, median of `reps` after one warm-up; the times include the op's host read. Entries = sum over the sources of
  the expansion X(s) = sum of d(w) over w in N(s); "longest run" = the largest common-neighbour count c among the sources' candidates,
  the length of the longest sequential sum.
Then recall@k on fb-pages-food seed 0: for every test positive (u, v), is v among u's top-k candidates (k = 20 / 50 / 100) on the
test split's graph, next to the AUC, hits@K and MRR of the same heuristics.      python tools/bench_recommend.py [reps]"""
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
from TwoWL.model.train import heuristic_scores, rank_scores, recommend
from TwoWL.operators.synthetic import rmat_edges
from twowl_b200 import ops

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 3
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


def expansion(ptr, adj, src):
    """X(s) for every source (int64, device)."""
    deg = ptr.diff()
    ds = deg[src]
    q = torch.repeat_interleave(torch.arange(src.numel(), device=dev), ds)
    first = torch.cumsum(ds, 0) - ds
    w = adj[ptr[src][q] + torch.arange(q.numel(), device=dev) - first[q]].long()
    return torch.zeros(src.numel(), dtype=torch.int64, device=dev).index_add_(0, q, deg[w])


def cuts(X, budget):
    """The op's batches: consecutive sources while the expansion stays within the budget, at least one each."""
    off = np.concatenate(([0], np.cumsum(X.cpu().numpy())))
    out, q = [], 0
    while q < X.numel():
        e = min(X.numel(), max(q + 1, int(np.searchsorted(off, off[q] + budget, side="right")) - 1))
        out.append((q, e))
        q = e
    return out


def torch_recommend(ptr, adj, keys, src, k, by, budget=1 << 25):
    """The same op in plain torch -> (ids [Q, k], fp32 scores [4, Q, k], aa float64 [Q, k])."""
    n, Q = ptr.numel() - 1, src.numel()
    deg = ptr.diff()
    ids = torch.full((Q, k), -1, dtype=torch.int64, device=dev)
    sc = torch.full((4, Q, k), float("nan"), device=dev)
    aa64 = torch.full((Q, k), float("nan"), dtype=torch.float64, device=dev)
    h = ops.HEURISTICS.index(by)
    for q0, q1 in cuts(expansion(ptr, adj, src), budget):
        qs = src[q0:q1]
        ds = deg[qs]
        j = torch.repeat_interleave(torch.arange(q1 - q0, device=dev), ds)
        first = torch.cumsum(ds, 0) - ds
        w = adj[ptr[qs][j] + torch.arange(j.numel(), device=dev) - first[j]].long()
        dw = deg[w]
        ej, ew = torch.repeat_interleave(j, dw), torch.repeat_interleave(w, dw)
        f2 = torch.cumsum(dw, 0) - dw
        t = torch.repeat_interleave(torch.arange(w.numel(), device=dev), dw)
        v = adj[ptr[w][t] + torch.arange(t.numel(), device=dev) - f2[t]].long()
        s = qs[ej]
        key = s * n + v
        pos = torch.searchsorted(keys, key).clamp_(max=max(keys.numel() - 1, 0))
        keep = (v != s) & (keys[pos] != key)
        qk = ej[keep] * n + v[keep]
        dwk = deg[ew[keep]].double()
        uq, inv, cnt = torch.unique(qk, sorted=True, return_inverse=True, return_counts=True)
        aa = torch.zeros(uq.numel(), dtype=torch.float64, device=dev).index_add_(0, inv, torch.where(dwk > 1, 1.0 / dwk.clamp(min=2).log(), 0.0))
        ra = torch.zeros(uq.numel(), dtype=torch.float64, device=dev).index_add_(0, inv, 1.0 / dwk)
        qv, vv = uq // n, uq % n
        cn = cnt.float()
        jac = cn / (ds[qv] + deg[vv] - cnt).float()
        rows = torch.stack((cn, jac, aa.float(), ra.float()))
        o = torch.sort(-rows[h], stable=True).indices                 # (q, v) order kept among equal scores
        o = o[torch.sort(qv[o], stable=True).indices]
        qo = qv[o]
        start = torch.cumsum(torch.bincount(qo, minlength=q1 - q0), 0) - torch.bincount(qo, minlength=q1 - q0)
        rank = torch.arange(o.numel(), device=dev) - start[qo]
        sel = rank < k
        r_q, r_k, r_o = q0 + qo[sel], rank[sel], o[sel]
        ids[r_q, r_k] = vv[r_o]
        sc[:, r_q, r_k] = rows[:, r_o]
        aa64[r_q, r_k] = aa[r_o]
    return ids, sc, aa64


def compare(ours, theirs, by, name):
    """ids equal for cn / jaccard; for aa / ra equal except at near-ties: the torch sums add the same terms in another order.
    cn / jaccard bits equal wherever the ids are. -> the number of near-tie swaps."""
    (i0, s0), (i1, s1, _) = ours, theirs
    assert torch.equal(i0 >= 0, i1 >= 0), f"{name}: candidate counts differ"
    same = (i0 == i1) & (i0 >= 0)
    assert torch.equal(s0[:2, same], s1[:2, same]), f"{name}: cn / jaccard differ"
    diff = i0 != i1
    if by in ("cn", "jaccard"):
        assert not bool(diff.any()), f"{name}: ids differ"
        return 0
    h = ops.HEURISTICS.index(by)        # where the ids differ, the two candidates' fp32 scores are within the bound of each other
    a, b = s0[h][diff].double(), s1[h][diff].double()
    c = torch.maximum(s0[0][diff], s1[0][diff]).double()
    r32 = torch.maximum(a, b).float()
    ulp = (torch.nextafter(r32, torch.full_like(r32, float("inf"))) - r32).double()
    assert bool(((a - b).abs() <= 2 * (0.5 * ulp + 2 * c * 2.0 ** -53 * r32.double()) + ulp).all()), f"{name}: {by} ids differ beyond near-ties"
    return int(diff.sum())


def row_keys(ptr, adj):
    n = ptr.numel() - 1
    return torch.repeat_interleave(torch.arange(n, device=dev), ptr.diff()) * n + adj.long()


def case(name, ptr, adj, keys, src, k, by):
    X = expansion(ptr, adj, src)
    entries = int(X.sum())
    nb = len(cuts(X, ops.RECOMMEND_MAX_ENTRIES))
    m0, m1, a, b = duel(lambda: ops.recommend_links(ptr, adj, src, k, by=by), lambda: torch_recommend(ptr, adj, keys, src, k, by))
    near = compare(a, b, by, name)
    print(f"{name:34s} by {by:7s} Q={src.numel():6d} entries={entries:13d} batches={nb:5d}  ours {m0:10.2f} ms "
          f"({entries / m0 / 1e6:7.3f} G entries/s)  torch {m1:10.2f} ms  x{m1 / m0:.1f}"
          + (f"  near-tie swaps {near}" if by in ("aa", "ra") else ""), flush=True)
    return a


# ---- R-MAT 1M / 16M: the test split's graph, 10^4 sources of test positives, and the hub alone
scale, samples, abcd, _ = bench.WORKLOADS["rmat"]
s, d, _ = rmat_edges(scale, samples, abcd, 0, dev)
bg = D.graph_from_split(D.do_edge_split(D._Data(torch.stack((s, d)))), pattern="none")   # no wedge index: no model here
bg.preprocess()
bg.setPosDegreeFeature()
tst = D.dataset(*bg.split(2))
n, E = bg.num_nodes, tst.ei.shape[1]
ptr, adj = ops.simple_adjacency(tst.ei[0], tst.ei[1], n)
deg = ptr.diff()
keys = row_keys(ptr, adj)
P = tst.y.shape[0] // 2
pos = tst.pos1[E::2][:P][tst.y.reshape(-1)[0::2] > 0.5]
src = pos[:10_000, 0].contiguous()
print(f"# R-MAT 1M/16M test split: n={n} nnz={adj.numel()} max deg={int(deg.max())}; default budget "
      f"{ops.RECOMMEND_MAX_ENTRIES} entries per batch", flush=True)
for by in ops.HEURISTICS:
    out = case("R-MAT 10^4 test-positive sources", ptr, adj, keys, src, 100, by)
    if by == "cn":
        print(f"{'':34s} longest run (largest c) = {int(out[1][0, :, 0].nan_to_num(0).max())}", flush=True)
hub = torch.argmax(deg).reshape(1)
for by in ("cn", "aa"):
    out = case(f"R-MAT hub alone (d = {int(deg.max())})", ptr, adj, keys, hub, 100, by)
    if by == "cn":
        print(f"{'':34s} longest run (largest c) = {int(out[1][0, 0, 0].nan_to_num(0))}", flush=True)
del bg, tst, ptr, adj, keys
torch.cuda.empty_cache()

# ---- fb-pages-food seed-0: recall@k of the held-out partner, next to the heuristics' AUC / hits@K / MRR
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
E = tst.ei.shape[1]
pos = tst.pos1[E::2][:labels.numel()][labels > 0.5]
print(f"# fb-pages-food seed 0, test split: {labels.numel()} pairs ({pos.shape[0]} positives); MRR over 100 filtered negatives; "
      f"recall@k = share of test positives (u, v) with v in u's top-k recommendations")
print(f"{'heuristic':10s} {'AUC':>8s} {'hits@20':>8s} {'hits@50':>8s} {'hits@100':>8s} {'MRR':>8s} {'rec@20':>8s} {'rec@50':>8s} {'rec@100':>8s}")
for name in ops.HEURISTICS:
    auc = float(ops.auc(h[name], labels)[0])
    hk = rank_scores(h[name], tst, (20, 50, 100))
    mrr = rank_scores(hr[name], rk, (20,))["mrr"]
    ids, _ = recommend(tst, pos[:, 0].contiguous(), k=100, by=name)
    hit = ids == pos[:, 1:2]
    rec = [float(hit[:, :kk].any(1).float().mean()) for kk in (20, 50, 100)]
    print(f"{name:10s} {auc:8.4f} {hk['hits@20']:8.4f} {hk['hits@50']:8.4f} {hk['hits@100']:8.4f} {mrr:8.4f} "
          f"{rec[0]:8.4f} {rec[1]:8.4f} {rec[2]:8.4f}", flush=True)
