"""Throughput of node2vec on the device (ops.node2vec_walks, ops.node2vec_step) and its link-prediction quality on fb-pages-food.
  Walks: R-MAT 1M nodes / 16M edge samples, the test split's graph (as tools/bench_global.py builds it), walks of length 80
    from 10^5 random starts (the isolated ones dropped), for (p, q) = (1, 1), (0.25, 4), (4, 0.25); walk steps per second against a torch-vectorised restatement
    of the same rejection sampler (all walks advance together; the neighbour test is torch.searchsorted on the sorted row * N + col
    keys). The torch version draws from torch's RNG, so its walks differ; the mean accepted trials per step are printed for both.
  Training: node2vec_step at d = 128 on the 1M-row table, batches of 1024 walks of length 20, window 5, K = 5 negatives per token;
    positive pairs per second over `batches` batches (one warm-up batch first), against nn.Embedding(sparse=True) +
    torch.optim.SparseAdam on the GPU fed the same walks and negatives. A full default epoch (10 walks per node of length 80,
    window 10) at R-MAT 1M is about 7.8e9 positive pairs plus as many negatives, 1.6e10 pairs in all: a count
    from the shapes.
  fb-pages-food seed 0, test split: AUC and hits@K of embedding_scores(node2vec_embedding) with 20 epochs of 128-walk batches (the
    default single epoch is only 7 Adam steps on its 620 nodes), next to CN, AA and
    PPR. The reference's recorded 0.8075 (logistic regression on node2vec features, BASELINE.md) is context only: its split and
    predictor differ.
CUDA-event times, median of `reps`.      python tools/bench_node2vec.py [reps] [batches]"""
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
from TwoWL.model.train import embedding_scores, global_heuristic_scores, heuristic_scores, node2vec_embedding, rank_scores
from TwoWL.operators.synthetic import rmat_edges
from twowl_b200 import ops

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 3
n_batches = int(sys.argv[2]) if len(sys.argv) > 2 else 20
dev = torch.device("cuda", 0)
try:
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True, timeout=60).stdout.strip()
except (OSError, subprocess.SubprocessError):
    card = ""
card = card or torch.cuda.get_device_name(dev) + " (power limit not read)"
print(f"# card: {card}", flush=True)


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


def torch_walks(ptr, adj, start, length, p, q, gen):
    """The same rejection sampler, every walk one lane of a torch vector -> (walks int64 [W, length], accepted trials)."""
    n = ptr.numel() - 1
    keys = torch.repeat_interleave(torch.arange(n, device=dev), ptr.diff()) * n + adj.long()   # sorted: rows, then sorted lists
    deg = ptr.diff()
    w_ret, w_in, w_out = 1 / p, 1.0, 1 / q
    wmax = max(w_ret, w_in, w_out)
    W = start.numel()
    out = torch.full((W, length), -1, dtype=torch.int64, device=dev)
    out[:, 0] = start
    cur, prev = start.clone(), torch.full_like(start, -1)
    trials = 0
    for t in range(1, length):
        live = deg[cur.clamp(min=0)] > 0
        live &= cur >= 0
        nxt = torch.full_like(cur, -1)
        todo = live.clone()
        while bool(todo.any()):
            idx = todo.nonzero().squeeze(1)
            c = cur[idx]
            x = adj[ptr[c] + (torch.rand(idx.numel(), device=dev, generator=gen) * deg[c]).long().clamp(max=deg[c] - 1)].long()
            trials += idx.numel()
            pv = prev[idx]
            if p == 1 and q == 1 or t == 1:
                acc = torch.ones_like(x, dtype=torch.bool)
            else:
                k = pv * n + x
                pos = torch.searchsorted(keys, k).clamp(max=keys.numel() - 1)
                w = torch.where(x == pv, w_ret, torch.where(keys[pos] == k, w_in, w_out))
                acc = torch.rand(idx.numel(), device=dev, generator=gen) * wmax < w
            nxt[idx[acc]] = x[acc]
            todo[idx[acc]] = False
        out[:, t] = nxt
        prev, cur = torch.where(live, cur, prev), nxt
    return out, trials


def torch_step(embm, opt, walks, negs, window):
    """The step's pairs and loss on nn.Embedding(sparse=True) + SparseAdam."""
    B, L = walks.shape
    K = negs.shape[2]
    w = walks.long()
    a_l, b_l = [], []
    for o in range(1, window + 1):
        a, b = w[:, :L - o].reshape(-1), w[:, o:].reshape(-1)
        m = (a >= 0) & (b >= 0)
        a_l.append(a[m])
        b_l.append(b[m])
    pa, pb = torch.cat(a_l), torch.cat(b_l)
    act = torch.zeros((B, L), dtype=torch.bool, device=dev)
    for o in range(1, window + 1):
        act[:, :L - o] |= (w[:, :L - o] >= 0) & (w[:, o:] >= 0)
    na = w[act].unsqueeze(1).expand(-1, K).reshape(-1)
    nb = negs[act].long().reshape(-1)
    opt.zero_grad()
    pos = (embm(pa) * embm(pb)).sum(-1)
    neg = (embm(na) * embm(nb)).sum(-1)
    loss = torch.nn.functional.softplus(-pos).mean() + torch.nn.functional.softplus(neg).mean()
    loss.backward()
    opt.step()
    return loss.detach(), pa.numel()


# ---- R-MAT 1M / 16M: the test split's graph
scale, samples, abcd, _ = bench.WORKLOADS["rmat"]
s, d, _ = rmat_edges(scale, samples, abcd, 0, dev)
bg = D.graph_from_split(D.do_edge_split(D._Data(torch.stack((s, d)))), pattern="none")
bg.preprocess()
bg.setPosDegreeFeature()
tst = D.dataset(*bg.split(2))
n = bg.num_nodes
ptr, adj = ops.simple_adjacency(tst.ei[0], tst.ei[1], n)
del bg, tst
torch.cuda.empty_cache()
print(f"# R-MAT 1M/16M test split: n={n} nnz={adj.numel()} max deg={int(ptr.diff().max())}", flush=True)

gen = torch.Generator(device=dev)
gen.manual_seed(0)
W, Lw = 100_000, 80
start = torch.randint(0, n, (W,), device=dev, generator=gen)
start = start[ptr.diff()[start] > 0]
for p, q in ((1.0, 1.0), (0.25, 4.0), (4.0, 0.25)):
    m0, m1, w0, (w1, tr1) = duel(lambda: ops.node2vec_walks(ptr, adj, start, Lw, p=p, q=q, seed=1),
                                 lambda: torch_walks(ptr, adj, start, Lw, p, q, gen))
    steps = int((w0[:, 1:] >= 0).sum())
    assert steps == start.numel() * (Lw - 1) and int((w1[:, 1:] >= 0).sum()) == steps
    print(f"walks p={p:4g} q={q:4g}: W={start.numel()} length={Lw}  ours {m0:8.2f} ms ({steps / (m0 * 1e-3) / 1e9:.3f} G steps/s)  "
          f"torch {m1:8.2f} ms ({steps / (m1 * 1e-3) / 1e9:.3f} G steps/s, {tr1 / steps:.3f} trials per step)  x{m1 / m0:.1f}",
          flush=True)

# ---- training: node2vec_step against SparseAdam on the same batches
d_, B, Lt, win, K = 128, 1024, 20, 5, 5
batches = []
for i in range(n_batches + 1):
    st = torch.randint(0, n, (B,), device=dev, generator=gen)
    batches.append((ops.node2vec_walks(ptr, adj, st, Lt, seed=2, index_base=i * B),
                    torch.randint(0, n, (B, Lt, K), device=dev, generator=gen, dtype=torch.int32)))
init = torch.randn((n, d_), device=dev, generator=gen)
emb, m, v, step = init.clone(), torch.zeros_like(init), torch.zeros_like(init), torch.zeros((), dtype=torch.int64, device=dev)
embm = torch.nn.Embedding(n, d_, sparse=True).to(dev)
with torch.no_grad():
    embm.weight.copy_(init)
opt = torch.optim.SparseAdam(embm.parameters(), lr=0.01)


def run_ours():
    return torch.stack([ops.node2vec_step(emb, m, v, step, w, ng, win) for w, ng in batches[1:]])


def run_torch():
    out = [torch_step(embm, opt, w, ng, win) for w, ng in batches[1:]]
    return torch.stack([o[0] for o in out]).double(), sum(o[1] for o in out)


ops.node2vec_step(emb, m, v, step, *batches[0], win)
torch_step(embm, opt, *batches[0], win)
t0, t1 = [], []
for _ in range(reps):
    ms, l0 = event_ms(run_ours)
    t0.append(ms)
    ms, (l1, npairs) = event_ms(run_torch)
    t1.append(ms)
m0, m1 = sorted(t0)[reps // 2], sorted(t1)[reps // 2]
print(f"step d={d_} B={B} L={Lt} window={win} K={K}: {n_batches} batches, {npairs} positive pairs (+ {K}/token negatives)  "
      f"ours {m0:8.2f} ms ({npairs / (m0 * 1e-3) / 1e6:.1f} M pos pairs/s)  torch SparseAdam {m1:8.2f} ms "
      f"({npairs / (m1 * 1e-3) / 1e6:.1f} M pos pairs/s)  x{m1 / m0:.1f}; first-pass losses ours {float(l0[0]):.4f} torch {float(l1[0]):.4f}",
      flush=True)
print(f"# a default epoch at this size: {n} x 10 walks x sum over i < 80 of min(10, 79 - i) = {n * 10 * sum(min(10, 79 - i) for i in range(80)):.3g} "
      f"positive pairs (a count from the shapes)", flush=True)
del emb, m, v, embm, opt, batches, ptr, adj
torch.cuda.empty_cache()

# ---- fb-pages-food seed 0
fb = np.load(os.path.join(ROOT, "tests", "golden", "fb_pages_food_seed0.npz"))
nf = int(fb["num_nodes"][0])
ep, en = (torch.from_numpy(fb[k].astype(np.int64)).to(dev) for k in ("edge_pos", "edge_neg"))
bg = D.BaseGraph(torch.zeros((nf, 0), device=dev), None, ep, en, torch.from_numpy(fb["num_pos"]), torch.from_numpy(fb["num_neg"]), "none")
bg.preprocess()
bg.setPosDegreeFeature()
tst = D.dataset(*bg.split(2))
labels = tst.y.reshape(-1)[0::2]
ms, (e, losses) = event_ms(lambda: node2vec_embedding(tst, epochs=20, batch_walks=128))
h = heuristic_scores(tst)
scores = {"node2vec": embedding_scores(tst, e), "cn": h["cn"], "aa": h["aa"], "ppr": global_heuristic_scores(tst, "ppr")}
print(f"# fb-pages-food seed 0, test split ({labels.numel()} pairs): node2vec (dim 128, 10 walks of 80 per node, window 10, "
      f"1 negative per positive, p = q = 1, 20 epochs of 128-walk batches) trained in {ms:.0f} ms, loss {losses[0]:.4f} -> {losses[-1]:.4f}")
print(f"{'score':10s} {'AUC':>8s} {'hits@20':>8s} {'hits@50':>8s} {'hits@100':>8s}")
for name, sc in scores.items():
    auc = float(ops.auc(sc, labels)[0])
    hk = rank_scores(sc, tst, (20, 50, 100))
    print(f"{name:10s} {auc:8.4f} {hk['hits@20']:8.4f} {hk['hits@50']:8.4f} {hk['hits@100']:8.4f}", flush=True)
print("reference (BASELINE.md): logistic regression on node2vec features, AUC 0.8075 - another split and predictor, context only")
