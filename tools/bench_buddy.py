"""Throughput of BUDDY on the device (ops.link_sketches, ops.sketch_features, train.buddy_fit / buddy_scores) and its link-prediction
quality on fb-pages-food.
  link_sketches: R-MAT 1M nodes / 16M edge samples, the test split's simple graph, hops 2, num_perm 128, hll_p 8. Time with the
    launches' host work included and gathered bytes per second: per hop nnz x (4 num_perm + m) bytes gathered from neighbours plus
    N rows read and written (gathered bytes, part of them served by L2: not DRAM traffic). Against a torch formulation
    (scatter_reduce amin / amax over the edge list), whose sketches must be equal.
  sketch_features: 10^5 random pairs, against a torch gather + compare formulation of the same estimator (float64), which must agree.
  One buddy_fit step on the training split at that scale (65 536 targets), by CUDA events: mask, sketches, features, fwd+bwd, Adam.
  buddy_scores over the test split.
  fb-pages-food seed 0: buddy trained on split 0 with the settings of tests/test_gpu_buddy.py: test AUC, hits@20/50/100, MRR against
    100 filtered negatives (ranking_dataset(bg, 2, 100)) and training seconds.
CUDA-event times, median of `reps`.      python tools/bench_buddy.py [reps]"""
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
from TwoWL.model.buddy import BUDDY
from TwoWL.model.train import _link_targets, buddy_fit, buddy_scores, rank_scores
from TwoWL.operators.synthetic import rmat_edges
from twowl_b200 import functional as F2
from twowl_b200 import graph, ops
from twowl_b200.optim import FusedAdam

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 3
BUDDY_FB = dict(epochs=40, batch_size=256, lr=5e-3, seed=0)   # the settings of tests/test_gpu_buddy.py
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


def torch_sketches(ptr, adj, hops, num_perm, hll_p, hop0):
    """The hops in plain torch: scatter_reduce amin (MinHash, as int64 of the uint32 bits) and amax (HyperLogLog, as int32) over
    the edge list, in edge chunks."""
    n = ptr.numel() - 1
    dst = torch.repeat_interleave(torch.arange(n, device=dev), ptr.diff())
    src = adj.long()
    mh = [hop0.minhash[0].long() & 0xFFFFFFFF]
    hl = [hop0.hll[0].int()]
    step = 1 << 21
    for _ in range(hops):
        m_out, h_out = mh[-1].clone(), hl[-1].clone()
        for e in range(0, src.numel(), step):
            s, d = src[e:e + step], dst[e:e + step]
            m_out.scatter_reduce_(0, d[:, None].expand(-1, num_perm), mh[-1][s], "amin", include_self=True)
            h_out.scatter_reduce_(0, d[:, None].expand(-1, 1 << hll_p), hl[-1][s], "amax", include_self=True)
        mh.append(m_out)
        hl.append(h_out)
    return torch.stack(mh).to(torch.int64), torch.stack(hl)


_THR = {4: 10.0, 5: 20.0, 6: 40.0, 7: 80.0, 8: 220.0, 9: 400.0, 10: 900.0}


def torch_est(M, p):
    m = float(1 << p)
    Z = torch.pow(2.0, -M.double()).sum(-1)
    V = (M == 0).sum(-1).double()
    alpha = {16.0: 0.673, 32.0: 0.697, 64.0: 0.709}.get(m, 0.7213 / (1.0 + 1.079 / m))
    lc = m * torch.log(m / V)
    return torch.where((V > 0) & (lc <= _THR[p]), lc, alpha * m * m / Z)


def torch_features(sk, u, v):
    k, P = sk.hops, u.numel()
    eu = torch.stack([torch_est(sk.hll[d][u], sk.hll_p) for d in range(k + 1)], 1)
    ev = torch.stack([torch_est(sk.hll[d][v], sk.hll_p) for d in range(k + 1)], 1)
    I = torch.zeros((P, k + 1, k + 1), dtype=torch.float64, device=dev)
    for a in range(1, k + 1):
        for b in range(1, k + 1):
            J = (sk.minhash[a][u] == sk.minhash[b][v]).sum(-1).double() / sk.num_perm
            I[:, a, b] = J * torch_est(torch.maximum(sk.hll[a][u], sk.hll[b][v]), sk.hll_p)
    A = (I[:, 1:, 1:] + I[:, :-1, :-1]) - (I[:, :-1, 1:] + I[:, 1:, :-1])
    Bu = (eu[:, 1:] - eu[:, :-1]) - A.sum(2)
    Bv = (ev[:, 1:] - ev[:, :-1]) - A.sum(1)
    return torch.cat((A.reshape(P, -1), Bu, Bv), 1).clamp(min=0).float()


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
nnz = adj.numel()
print(f"# R-MAT 1M/16M test split: n={n} nnz={nnz} max deg={int(ptr.diff().max())}", flush=True)
K, NP, HP = 2, 128, 8
row = 4 * NP + (1 << HP)
ms, sk = median_ms(lambda: ops.link_sketches(ptr, adj, K, NP, HP))
gathered = K * (nnz * row + 2 * n * row)
t_ms, (tm, th) = median_ms(lambda: torch_sketches(ptr, adj, K, NP, HP, sk))
assert torch.equal(sk.minhash.long() & 0xFFFFFFFF, tm) and torch.equal(sk.hll.int(), th), "sketches differ from the torch formulation"
print(f"link_sketches hops {K}, num_perm {NP}, hll_p {HP}: {ms:.2f} ms, {gathered / 1e9:.2f} GB gathered, "
      f"{gathered / ms / 1e9:.2f} TB/s gathered; torch scatter_reduce {t_ms:.1f} ms, ratio {t_ms / ms:.1f}x; sketches equal", flush=True)
del tm, th
g = torch.Generator(device="cpu").manual_seed(1)
qs = torch.randint(0, n, (100000, 2), generator=g).to(dev)
ms, f = median_ms(lambda: ops.sketch_features(sk, qs[:, 0], qs[:, 1]))
sk64 = ops.LinkSketches(sk.minhash.long() & 0xFFFFFFFF, sk.hll, K, NP, HP, 0)
t_ms, tf = median_ms(lambda: torch_features(sk64, qs[:, 0], qs[:, 1]))
err = float(((f - tf).abs() / tf.abs().clamp(min=1.0)).max())
assert err < 1e-5, f"features differ from the torch formulation: {err}"
print(f"sketch_features 10^5 random pairs: {ms:.3f} ms, {1e5 / ms * 1e3:.3e} pairs/s; torch gather + compare {t_ms:.1f} ms, "
      f"ratio {t_ms / ms:.1f}x; max relative difference {err:.1e}", flush=True)
del sk, sk64, f, tf
torch.cuda.empty_cache()

# ---- one buddy_fit step at that scale, by phase
N = trn.x.shape[0]
tptr, tadj = graph.simple_adjacency(trn.ei, N)
pairs, y = _link_targets(trn)
n_pos = trn.ei.shape[1] // 2
torch.manual_seed(0)
mod = BUDDY(K, 0.5).to(dev).train()
opt = FusedAdam(mod.parameters(), lr=1e-3)
perm = torch.randperm(pairs.shape[0], generator=torch.Generator(device="cpu").manual_seed(0)).to(dev)
phases = {"mask": [], "sketches": [], "features": [], "fwd+bwd": [], "adam": [], "step": []}
for it in range(reps + 1):
    ids = perm[it * 65536:(it + 1) * 65536]
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
    ev[0].record()
    bp = pairs[ids]
    pos = ids[ids < n_pos]
    mask = ops.adjacency_pair_mask(tptr, tadj, pairs[pos, 0], pairs[pos, 1])
    ev[1].record()
    tsk = ops.link_sketches(tptr, tadj, K, NP, HP, entry_mask=mask)
    ev[2].record()
    sf = ops.sketch_features(tsk, bp[:, 0], bp[:, 1])
    ev[3].record()
    opt.zero_grad()
    loss = F2.bce_with_logits(mod(sf, seed=it), y[ids].unsqueeze(-1))
    loss.backward()
    ev[4].record()
    opt.step()
    ev[5].record()
    torch.cuda.synchronize()
    if it:
        for i, k_ in enumerate(("mask", "sketches", "features", "fwd+bwd", "adam")):
            phases[k_].append(ev[i].elapsed_time(ev[i + 1]))
        phases["step"].append(ev[0].elapsed_time(ev[5]))
print(f"buddy_fit step, R-MAT 1M/16M training split ({tadj.numel()} adjacency entries), 65536 targets, hops {K}: "
      + ", ".join(f"{k} {np.median(v):.2f} ms" for k, v in phases.items()), flush=True)
mod.eval()
ms, sc = median_ms(lambda: buddy_scores(mod, tst))
print(f"buddy_scores, R-MAT test split: {sc.numel()} pairs in {ms:.1f} ms, {sc.numel() / ms * 1e3:.3e} pairs/s (sketching included)",
      flush=True)
del trn, tst, tptr, tadj, ptr, adj, mod, opt, pairs, y, perm, sc, tsk, mask
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
torch.cuda.synchronize()
t0 = time.perf_counter()
m, losses = buddy_fit(trn, **BUDDY_FB)
torch.cuda.synchronize()
secs = time.perf_counter() - t0
s_, r_ = buddy_scores(m, tst), buddy_scores(m, rds)
rk = rank_scores(s_, tst, (20, 50, 100))
mrr = rank_scores(r_, rds, (20,))["mrr"]
print(f"# fb-pages-food seed 0 test split; buddy: {BUDDY_FB}, hops 2, num_perm 128, hll_p 8")
print(f"fb-pages-food test buddy: AUC {float(ops.auc(s_, labels)[0]):.4f} " + " ".join(f"{k} {v:.4f}" for k, v in rk.items())
      + f" mrr(100 filtered) {mrr:.4f} train {secs:.2f} s", flush=True)
