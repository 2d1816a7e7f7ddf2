"""Throughput of NCN on the device (ops.common_neighbors, TwoWL.model.ncn.NCN, train.ncn_scores) and its link-prediction quality on
fb-pages-food.
  common_neighbors: R-MAT 1M nodes / 16M edge samples, the test split's graph (as tools/bench_seal.py builds it), for 10^5 random
    pairs and for 10^4 test positives plus 10^4 test negatives. Time with the host reads included, entries and entries/s, against a
    torch formulation of the same intersection (tools/bench_heuristics.py's probe by searchsorted), whose lists must be equal.
  One ncn_fit step on the training split at that scale (hidden 64, 2 layers, 65 536 targets), split by CUDA events into encoder
    forward + backward, mask + common-neighbour extraction, predictor forward + backward, and the Adam step.
  ncn_scores over the test split: pairs per second (one encoder pass included).
  fb-pages-food seed 0: ncn and gcn (cn=False) trained on split 0 with the settings of tests/test_gpu_ncn.py, next to seal / cn / aa
    / ppr / node2vec: test AUC, hits@20/50/100 (rank_scores), MRR against 100 filtered negatives (ranking_dataset(bg, 2, 100)) and
    training seconds.
CUDA-event times, median of `reps`.      python tools/bench_ncn.py [reps]"""
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "link-prediction-gnn_b200")):
    sys.path.insert(0, p)
import numpy as np
import torch

import bench
import TwoWL.operators.datasets as D
from TwoWL.model.ncn import NCN
from TwoWL.model.train import _link_targets, embedding_scores, global_heuristic_scores, heuristic_scores, ncn_fit, ncn_scores, \
    node2vec_embedding, rank_scores, seal_fit, seal_scores
from TwoWL.operators.synthetic import rmat_edges
from TwoWL.utils import double, sample_block
from twowl_b200 import functional as F2
from twowl_b200 import graph, ops
from twowl_b200.optim import FusedAdam

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 3
NCN_FB = dict(epochs=40, batch_size=256, lr=5e-3, seed=0)   # the settings of tests/test_gpu_ncn.py
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


def median_ms(fn):
    fn()
    ts = []
    for _ in range(reps):
        t, out = event_ms(fn)
        ts.append(t)
    return float(np.median(ts)), out


def torch_lists(keys, ptr, adj, u, v):
    """The common-neighbour lists in plain torch: the shorter list of each pair expanded, probed by searchsorted into the sorted
    (row, neighbour) keys -> (cn_ptr, ids)."""
    n, P = ptr.numel() - 1, u.numel()
    deg = ptr.diff()
    du, dv = deg[u], deg[v]
    swap = (du > dv) | ((du == dv) & (u > v))
    s, l_ = torch.where(swap, v, u), torch.where(swap, u, v)
    ds = deg[s]
    pair = torch.repeat_interleave(torch.arange(P, device=dev), ds)
    first = torch.cumsum(ds, 0) - ds
    x = adj[ptr[s][pair] + torch.arange(pair.numel(), device=dev) - first[pair]].long()
    q = l_[pair] * n + x
    pos = torch.searchsorted(keys, q).clamp_(max=max(keys.numel() - 1, 0))
    hit = keys[pos] == q
    cnt = torch.bincount(pair[hit], minlength=P)
    return torch.cat((cnt.new_zeros(1), torch.cumsum(cnt, 0))), x[hit].to(torch.int32)


def compare_cn(name, u, v):
    ours_ms, cn = median_ms(lambda: ops.common_neighbors(ptr, adj, u, v))
    theirs_ms, (tp, ti) = median_ms(lambda: torch_lists(keys, ptr, adj, u, v))
    assert torch.equal(cn.ptr, tp) and torch.equal(cn.ids, ti), f"{name}: lists differ from the torch formulation"
    nnz = cn.ids.numel()
    print(f"common_neighbors {name}: {u.numel()} pairs, {nnz} entries in {ours_ms:.2f} ms ({nnz / ours_ms * 1e3:.3e} entries/s, "
          f"{u.numel() / ours_ms * 1e3:.3e} pairs/s); torch formulation {theirs_ms:.2f} ms, ratio {theirs_ms / ours_ms:.1f}x; "
          f"lists equal", flush=True)


# ---- R-MAT 1M / 16M
scale, samples, abcd, _ = bench.WORKLOADS["rmat"]
s, d, _ = rmat_edges(scale, samples, abcd, 0, dev)
bg = D.graph_from_split(D.do_edge_split(D._Data(torch.stack((s, d)))), pattern="none")
bg.preprocess()
bg.setPosDegreeFeature()
trn, tst = D.dataset(*bg.split(0)), D.dataset(*bg.split(2))
n = bg.num_nodes
del bg
ptr, adj = graph.simple_adjacency(tst.ei, n)
rows = torch.repeat_interleave(torch.arange(n, device=dev), ptr.diff())
keys = rows * n + adj.long()
del rows
print(f"# R-MAT 1M/16M test split: n={n} nnz={adj.numel()} max deg={int(ptr.diff().max())}", flush=True)
g = torch.Generator(device="cpu").manual_seed(1)
qs = torch.randint(0, n, (100000, 2), generator=g).to(dev)
compare_cn("random pairs", qs[:, 0], qs[:, 1])
E = tst.ei.shape[1]
tp_ = tst.pos1[E::2][: tst.y.shape[0] // 2].to(torch.long)
lab = tst.y.reshape(-1)[0::2][: tp_.shape[0]] > 0.5
sel = torch.cat((tp_[lab][:10000], tp_[~lab][:10000]))
compare_cn("test positives + negatives", sel[:, 0], sel[:, 1])
del keys
torch.cuda.empty_cache()

# ---- one ncn_fit step at that scale, by phase
N = trn.x.shape[0]
tptr, tadj = graph.simple_adjacency(trn.ei, N)
pairs, y = _link_targets(trn)
n_pos = trn.ei.shape[1] // 2
torch.manual_seed(0)
mod = NCN(int(trn.x.max()), 64, 2, 0.3).to(dev).train()
opt = FusedAdam(mod.parameters(), lr=1e-3)
perm = torch.randperm(pairs.shape[0], generator=torch.Generator(device="cpu").manual_seed(0)).to(dev)
phases = {"sample_block + encoder fwd+bwd": [], "mask + CN extraction": [], "predictor fwd+bwd": [], "adam": [], "step": []}
for it in range(reps + 1):
    ids = perm[it * 65536:(it + 1) * 65536]
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(7)]
    ev[0].record()
    bp = pairs[ids]
    pos = ids[ids < n_pos]
    ei_new, x_new, _ = sample_block(double(pos, for_index=True), N, trn.ei, None)
    opt.zero_grad()
    h = mod.encode(x_new, ei_new, None, seed=it)
    ev[1].record()
    cn = ops.common_neighbors(tptr, tadj, bp[:, 0], bp[:, 1], ops.adjacency_pair_mask(tptr, tadj, pairs[pos, 0], pairs[pos, 1]))
    ev[2].record()
    hd = h.detach().requires_grad_()
    loss = F2.bce_with_logits(mod.predict(hd, bp, cn, seed=it), y[ids].unsqueeze(-1))
    loss.backward()
    ev[3].record()
    h.backward(hd.grad)
    ev[4].record()
    opt.step()
    ev[5].record()
    torch.cuda.synchronize()
    if it:
        phases["sample_block + encoder fwd+bwd"].append(ev[0].elapsed_time(ev[1]) + ev[3].elapsed_time(ev[4]))
        phases["mask + CN extraction"].append(ev[1].elapsed_time(ev[2]))
        phases["predictor fwd+bwd"].append(ev[2].elapsed_time(ev[3]))
        phases["adam"].append(ev[4].elapsed_time(ev[5]))
        phases["step"].append(ev[0].elapsed_time(ev[5]))
print(f"ncn_fit step, R-MAT 1M/16M training split ({trn.ei.shape[1]} directed edges), 65536 targets, hidden 64, 2 layers, "
      f"{cn.ids.numel()} CN entries: " + ", ".join(f"{k} {np.median(v):.2f} ms" for k, v in phases.items()), flush=True)
mod.eval()
ms, sc = median_ms(lambda: ncn_scores(mod, tst))
print(f"ncn_scores, R-MAT test split: {sc.numel()} pairs in {ms:.1f} ms, {sc.numel() / ms * 1e3:.3e} pairs/s", flush=True)
del trn, tst, tptr, tadj, ptr, adj, mod, opt, pairs, y, perm, sc, cn, h, hd
graph.clear_cache()
torch.cuda.empty_cache()

# ---- fb-pages-food seed 0
fb = np.load(os.path.join(ROOT, "tests", "golden", "fb_pages_food_seed0.npz"))
nf = int(fb["num_nodes"][0])
ep, en = (torch.from_numpy(fb[k].astype(np.int64)).to(dev) for k in ("edge_pos", "edge_neg"))
bg = D.BaseGraph(torch.zeros((nf, 0), device=dev), None, ep, en, torch.from_numpy(fb["num_pos"]), torch.from_numpy(fb["num_neg"]), "none")
bg.preprocess()
bg.setPosDegreeFeature()
trn, tst = D.dataset(*bg.split(0)), D.dataset(*bg.split(2))
rds = D.ranking_dataset(bg, 2, num_neg=100)
labels = tst.y.reshape(-1)[0::2]


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, out


rows_ = {}
for name, cn_term in (("ncn", True), ("gcn", False)):
    secs, (m, _) = timed(lambda: ncn_fit(trn, cn=cn_term, **NCN_FB))
    rows_[name] = (secs, ncn_scores(m, tst), ncn_scores(m, rds))
secs, (m, _) = timed(lambda: seal_fit(trn, 10, 32, lr=1e-3, hops=1, seed=0))
rows_["seal"] = (secs, seal_scores(m, tst), seal_scores(m, rds))
for k in ("cn", "aa"):
    rows_[k] = (0.0, heuristic_scores(tst)[k], heuristic_scores(rds)[k])
rows_["ppr"] = (0.0, global_heuristic_scores(tst, "ppr"), global_heuristic_scores(rds, "ppr"))
secs, (emb, _) = timed(lambda: node2vec_embedding(tst, epochs=20, batch_walks=128))
rows_["node2vec"] = (secs, embedding_scores(tst, emb), embedding_scores(rds, emb))
print(f"# fb-pages-food seed 0 test split; ncn / gcn: {NCN_FB}")
for name, (secs, s_, r_) in rows_.items():
    rk = rank_scores(s_, tst, (20, 50, 100))
    mrr = rank_scores(r_, rds, (20,))["mrr"]
    print(f"fb-pages-food test {name}: AUC {float(ops.auc(s_, labels)[0]):.4f} " + " ".join(f"{k} {v:.4f}" for k, v in rk.items())
          + f" mrr(100 filtered) {mrr:.4f} train {secs:.2f} s", flush=True)
