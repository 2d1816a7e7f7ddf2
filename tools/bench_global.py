"""Time of the global link-prediction heuristics (ops.global_heuristics, ops.recommend_global) and their retrieval on fb-pages-food.
  R-MAT 1M nodes / 16M edge samples, the test split's message-passing graph (train + val edges):
    Katz (3 steps, beta 0.001): the first 10^4 test positives as pairs (their distinct sources are the walks), and recommendations
      k = 100 for their sources;
    PPR (20 steps, alpha 0.85): the same for the first 10^3 test positives (20 propagation steps per batch instead of 3);
  each against a plain torch formulation, alternating in one process: torch.sparse CSR (values = the per-node scale of the source
  column) @ a dense fp32 [N, B] operand with the same recursion and batch width, then a gather, or topk over each column with s and
  N(s) masked. Scores must agree within the tests' a-priori bound (cuSPARSE adds in another order); ids may differ only where the
  two candidates' scores lie within that bound (torch's tie order is unspecified).
  CUDA-event time, median of `reps` after one warm-up; the times include the ops' host read. "gathered" = the bytes seg_reduce
  gathers per propagation step, nnz x operand width x 4, and the rate is that over the op's time per step (steps x batches).
  Then recommend_global at max_cols 64 / 128 / 256, the choice of the default.
Then fb-pages-food seed 0: AUC / hits@K / MRR of katz and ppr next to the four local heuristics, recall@20/50/100 of the held-out
test partner by recommend_global next to recommend_links, and the share of test positives whose partner lies within two hops,
three hops and in the source's component of the test split's graph.      python tools/bench_global.py [reps]"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "link-prediction-gnn_b200")):
    sys.path.insert(0, p)
import numpy as np
import scipy.sparse as sp
import scipy.sparse.csgraph as csg
import torch

import bench
import TwoWL.operators.datasets as D
from TwoWL.model.train import global_heuristic_scores, heuristic_scores, rank_scores, recommend, recommend_global
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


def timed(fn):
    """`reps` runs after one warm-up -> (median ms, result)."""
    out = fn()
    t = []
    for _ in range(reps):
        ms, out = event_ms(fn)
        t.append(ms)
    return sorted(t)[reps // 2], out


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


def bound(ptr, steps):
    u = 2.0 ** -24
    m = int(ptr.diff().max()) + 2
    return (1 + m * u / (1 - m * u)) ** steps - 1


class TorchWalk:
    """The same recursion on torch.sparse: A_scaled[v, w] = scale[w], one dense [N, B] operand per batch of sources."""

    def __init__(self, ptr, adj, by, steps, damping):
        n = ptr.numel() - 1
        d = ptr.diff().float()
        p = torch.tensor(damping, dtype=torch.float32, device=dev)
        scale = torch.full((n,), float(p), device=dev) if by == "katz" else torch.where(d > 0, p / d.clamp(min=1), 0.0)
        self.A = torch.sparse_csr_tensor(ptr, adj.long(), scale[adj.long()], (n, n))
        self.n, self.by, self.steps, self.restart = n, by, steps, float(torch.tensor(1.0) - p)

    def run(self, src):
        B = src.numel()
        cols = torch.arange(B, device=dev)
        Y = torch.zeros((self.n, B), device=dev)
        if self.by == "ppr":
            Y[src, cols] += 1.0
        for _ in range(self.steps):
            if self.by == "katz":
                Y[src, cols] += 1.0
            Y = self.A @ Y
            if self.by == "ppr":
                Y[src, cols] += self.restart
        return Y


def torch_pairs(tw, u, v, cols):
    us, inv = torch.unique(u, return_inverse=True)
    out = torch.empty(u.numel(), device=dev)
    for c0 in range(0, us.numel(), cols):
        Y = tw.run(us[c0:c0 + cols])
        m = (inv >= c0) & (inv < c0 + cols)
        out[m] = Y[v[m], inv[m] - c0]
    return out


def torch_topk(tw, ptr, adj, src, k, cols):
    n = ptr.numel() - 1
    ids = torch.full((src.numel(), k), -1, dtype=torch.int64, device=dev)
    sc = torch.full((src.numel(), k), float("nan"), device=dev)
    deg = ptr.diff()
    for q0 in range(0, src.numel(), cols):
        s = src[q0:q0 + cols]
        Y = tw.run(s)
        j = torch.repeat_interleave(torch.arange(s.numel(), device=dev), deg[s])
        first = torch.cumsum(deg[s], 0) - deg[s]
        nb = adj[ptr[s][j] + torch.arange(j.numel(), device=dev) - first[j]].long()
        Y[nb, j] = 0.0
        Y[s, torch.arange(s.numel(), device=dev)] = 0.0
        Y = torch.where(Y > 0, Y, float("-inf"))
        kk = min(k, n)
        val, idx = torch.topk(Y.t(), kk, dim=1)
        ok = val > float("-inf")
        ids[q0:q0 + s.numel(), :kk] = torch.where(ok, idx, -1)
        sc[q0:q0 + s.numel(), :kk] = torch.where(ok, val, float("nan"))
    return ids, sc


def close(a, b, tol):
    """|a - b| within the bound of both against the exact value, plus the underflow floor."""
    a, b = a.double(), b.double()
    return (a - b).abs() <= 2 * tol * torch.maximum(a, b) + 8 * 2.0 ** -126


def run_method(name, by, steps, damping, ptr, adj, pos, n_pairs):
    cols = ops.WALK_MAX_COLS
    nnz = adj.numel()
    u, v = pos[:n_pairs, 0].contiguous(), pos[:n_pairs, 1].contiguous()
    U = int(torch.unique(u).numel())
    tol = bound(ptr, steps)
    tw = TorchWalk(ptr, adj, by, steps, damping)
    width = max(68, cols)
    per_step = nnz * width * 4
    m0, m1, a, b = duel(lambda: ops.global_heuristics(ptr, adj, u, v, by=by, steps=steps, damping=damping),
                        lambda: torch_pairs(tw, u, v, cols))
    assert bool(close(a, b, tol).all()), f"{name}: pair scores differ beyond the bound"
    nsteps = steps * -(-U // cols)
    print(f"{name:5s} pairs  P={n_pairs:6d} sources={U:6d} batches={-(-U // cols):4d} x {steps:2d} steps  ours {m0:9.2f} ms "
          f"({per_step / 1e9:.2f} GB gathered per step, {per_step * nsteps / (m0 * 1e-3) / 1e12:.2f} TB/s)  torch {m1:9.2f} ms  "
          f"x{m1 / m0:.2f}", flush=True)
    src = u
    m0, m1, (i0, s0), (i1, s1) = duel(lambda: ops.recommend_global(ptr, adj, src, 100, by=by, steps=steps, damping=damping),
                                      lambda: torch_topk(tw, ptr, adj, src, 100, cols))
    same = (i0 == i1) & (i0 >= 0)
    assert bool(close(s0[same], s1[same], tol).all()), f"{name}: top-k scores differ beyond the bound"
    diff = (i0 != i1) & (i0 >= 0) & (i1 >= 0)
    assert bool(close(s0[diff], s1[diff], tol).all()), f"{name}: top-k ids differ beyond near-ties"
    nsteps = steps * -(-src.numel() // cols)
    print(f"{name:5s} top-100 Q={src.numel():6d} batches={-(-src.numel() // cols):4d} x {steps:2d} steps  ours {m0:9.2f} ms "
          f"({per_step * nsteps / (m0 * 1e-3) / 1e12:.2f} TB/s gathered)  torch {m1:9.2f} ms  x{m1 / m0:.2f}  "
          f"near-tie id swaps {int(diff.sum())}, rows with fewer valid ids than torch {int(((i0 >= 0).sum(1) != (i1 >= 0).sum(1)).sum())}",
          flush=True)
    return src


# ---- R-MAT 1M / 16M: the test split's graph
scale, samples, abcd, _ = bench.WORKLOADS["rmat"]
s, d, _ = rmat_edges(scale, samples, abcd, 0, dev)
bg = D.graph_from_split(D.do_edge_split(D._Data(torch.stack((s, d)))), pattern="none")   # no wedge index: no model here
bg.preprocess()
bg.setPosDegreeFeature()
tst = D.dataset(*bg.split(2))
n, E = bg.num_nodes, tst.ei.shape[1]
ptr, adj = ops.simple_adjacency(tst.ei[0], tst.ei[1], n)
P = tst.y.shape[0] // 2
pos = tst.pos1[E::2][:P][tst.y.reshape(-1)[0::2] > 0.5]
del bg, tst
torch.cuda.empty_cache()
print(f"# R-MAT 1M/16M test split: n={n} nnz={adj.numel()} max deg={int(ptr.diff().max())}; {ops.WALK_MAX_COLS} sources per batch "
      f"(operand width {max(68, ops.WALK_MAX_COLS)}), k = 100", flush=True)
run_method("katz", "katz", 3, 0.001, ptr, adj, pos, 10_000)
src = run_method("ppr", "ppr", 20, 0.85, ptr, adj, pos, 1_000)
for cols in (64, 128, 256):
    ms, _ = timed(lambda: ops.recommend_global(ptr, adj, src, 100, by="ppr", max_cols=cols))
    print(f"ppr top-100 Q={src.numel()} max_cols={cols:4d}: {ms:9.2f} ms", flush=True)
del ptr, adj, pos
torch.cuda.empty_cache()

# ---- fb-pages-food seed-0: the global heuristics next to the local ones
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
for by in ops.GLOBAL_HEURISTICS:
    h[by], hr[by] = global_heuristic_scores(tst, by), global_heuristic_scores(rk, by)
labels = tst.y.reshape(-1)[0::2]
E = tst.ei.shape[1]
pos = tst.pos1[E::2][:labels.numel()][labels > 0.5]
print(f"# fb-pages-food seed 0, test split: {labels.numel()} pairs ({pos.shape[0]} positives); MRR over 100 filtered negatives; "
      f"recall@k = share of test positives (u, v) with v in u's top-k recommendations (recommend_links for the local heuristics, "
      f"recommend_global for katz / ppr)")
print(f"{'heuristic':10s} {'AUC':>8s} {'hits@20':>8s} {'hits@50':>8s} {'hits@100':>8s} {'MRR':>8s} {'rec@20':>8s} {'rec@50':>8s} {'rec@100':>8s}")
for name in ops.HEURISTICS + ops.GLOBAL_HEURISTICS:
    auc = float(ops.auc(h[name], labels)[0])
    hk = rank_scores(h[name], tst, (20, 50, 100))
    mrr = rank_scores(hr[name], rk, (20,))["mrr"]
    fn = recommend_global if name in ops.GLOBAL_HEURISTICS else recommend
    ids = fn(tst, pos[:, 0].contiguous(), k=100, by=name)[0]
    hit = ids == pos[:, 1:2]
    rec = [float(hit[:, :kk].any(1).float().mean()) for kk in (20, 50, 100)]
    print(f"{name:10s} {auc:8.4f} {hk['hits@20']:8.4f} {hk['hits@50']:8.4f} {hk['hits@100']:8.4f} {mrr:8.4f} "
          f"{rec[0]:8.4f} {rec[1]:8.4f} {rec[2]:8.4f}", flush=True)
# the recall ceilings: hop distance from each test positive's source to its partner on the test split's graph
ei = tst.ei.cpu().numpy()
A = sp.csr_matrix((np.ones(ei.shape[1]), (ei[0], ei[1])), shape=(nf, nf))
A = ((A + A.T) > 0).astype(np.float64)
pu, pv = pos[:, 0].cpu().numpy(), pos[:, 1].cpu().numpy()
dist = csg.shortest_path(A, unweighted=True, indices=np.unique(pu))
row = {s: i for i, s in enumerate(np.unique(pu))}
dd = dist[[row[x] for x in pu], pv]
iso = np.asarray(A.sum(1)).ravel()[pu] == 0
print(f"ceilings over {pu.size} test positives: within two hops {np.mean(dd <= 2):.4f}, within three hops {np.mean(dd <= 3):.4f}, "
      f"same component {np.mean(np.isfinite(dd)):.4f}; isolated source {np.mean(iso):.4f}", flush=True)
