"""Throughput of SEAL on the device (ops.seal_subgraphs, TwoWL.model.seal.DGCNN) and its link-prediction quality on fb-pages-food.
  Extraction: R-MAT 1M nodes / 16M edge samples, the test split's graph (as tools/bench_global.py builds it), 10^5 random query
    pairs; 1 hop with max_nodes_per_hop 100 and 2 hops with 50. Subgraphs per second and labelled nodes per second (count + fill,
    host read included), against a numpy / scipy restatement of the same rule (layers by np.unique, the cap by the same hash,
    induced edges by np.isin, DRNL by scipy's shortest_path) on the first `host_q` queries.
  DGCNN: forward + backward of one batch of 1024 of those 1-hop subgraphs (k = 30, hidden 32, 3 layers), extraction excluded.
  fb-pages-food seed 0: seal_fit on split 0 (10 epochs, batches of 32, lr 1e-3, 1 hop, no cap), wall time, then the test split's AUC
    and hits@K of seal_scores, next to CN, AA and PPR.
CUDA-event times, median of `reps`.      python tools/bench_seal.py [reps] [host_q]"""
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "link-prediction-gnn_b200")):
    sys.path.insert(0, p)
import numpy as np
import scipy.sparse as sp
from scipy.sparse.csgraph import shortest_path
import torch

import bench
import TwoWL.operators.datasets as D
from TwoWL.model.seal import DGCNN
from TwoWL.model.train import global_heuristic_scores, heuristic_scores, rank_scores, seal_fit, seal_scores
from TwoWL.operators.synthetic import rmat_edges
from twowl_b200 import ops

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 3
host_q = int(sys.argv[2]) if len(sys.argv) > 2 else 200
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


M64 = np.uint64(0xFFFFFFFFFFFFFFFF)


def np_hash(seed, idx):
    """hash_u32 of common.cuh over a uint64 array."""
    with np.errstate(over="ignore"):
        z = idx + np.uint64(seed) * np.uint64(0x9E3779B97F4A7C15) + np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return (z ^ (z >> np.uint64(31))) >> np.uint64(32)


def host_subgraph(hp, ha, u, v, hops, cap, seed, q):
    nodes = [np.array([min(u, v), max(u, v)], np.int64)]
    seen = nodes[0]
    fringe = nodes[0]
    for _ in range(hops):
        nb = np.concatenate([ha[hp[x]:hp[x + 1]] for x in fringe]) if fringe.size else np.zeros(0, np.int32)
        cand = np.setdiff1d(np.unique(nb), seen)
        seen = np.union1d(seen, cand)
        if cap and cand.size > cap:
            h = np_hash(seed, (np.uint64(q) << np.uint64(32)) | cand.astype(np.uint64))
            cand = cand[np.lexsort((cand, h))[:cap]]
        fringe = cand
        nodes.append(cand)
    nodes = np.sort(np.concatenate(nodes))
    rows = np.repeat(np.arange(nodes.size), hp[nodes + 1] - hp[nodes])
    cols = np.concatenate([ha[hp[x]:hp[x + 1]] for x in nodes])
    keep = np.isin(cols, nodes)
    rows, cols = rows[keep], np.searchsorted(nodes, cols[keep])
    lu, lv = np.searchsorted(nodes, u), np.searchsorted(nodes, v)
    keep = ~(((rows == lu) & (cols == lv)) | ((rows == lv) & (cols == lu)))
    A = sp.csr_matrix((np.ones(int(keep.sum())), (rows[keep], cols[keep])), shape=(nodes.size, nodes.size))
    m = np.ones(nodes.size, bool)
    m[lv] = False
    du = np.full(nodes.size, np.inf)
    du[m] = shortest_path(A[m][:, m], unweighted=True, indices=int(m[:lu].sum()))
    m[lv], m[lu] = True, False
    dv = np.full(nodes.size, np.inf)
    dv[m] = shortest_path(A[m][:, m], unweighted=True, indices=int(m[:lv].sum()))
    return nodes, du, dv


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
g = torch.Generator(device="cpu").manual_seed(1)
Q = 100000
qs = torch.randint(0, n, (Q, 2), generator=g)
qs = qs[qs[:, 0] != qs[:, 1]].to(dev)
hp, ha = ptr.cpu().numpy(), adj.cpu().numpy()
host_pairs = qs[:host_q].cpu().numpy()
sub1 = None
for hops, cap in ((1, 100), (2, 50)):
    ms, sub = median_ms(lambda: ops.seal_subgraphs(ptr, adj, qs[:, 0], qs[:, 1], hops=hops, max_nodes_per_hop=cap, seed=0))
    if hops == 1:
        sub1 = sub
    nq, nn_, ne = qs.shape[0], sub.nodes.numel(), sub.edge_index.shape[1]
    t0 = time.perf_counter()
    for i, (u, v) in enumerate(host_pairs.tolist()):
        host_subgraph(hp, ha, u, v, hops, cap, 0, i)
    host_s = time.perf_counter() - t0
    print(f"extract hops={hops} cap={cap}: {nq} subgraphs, {nn_} nodes, {ne} edges in {ms:.1f} ms: {nq / ms * 1e3:.3e} subgraphs/s, "
          f"{nn_ / ms * 1e3:.3e} labelled nodes/s; host restatement {host_pairs.shape[0] / host_s:.3e} subgraphs/s "
          f"({host_pairs.shape[0]} queries), ratio {nq / ms * 1e3 / (host_pairs.shape[0] / host_s):.0f}x", flush=True)

# ---- DGCNN forward + backward on 1024 of the 1-hop subgraphs
sub = ops.seal_subgraphs(ptr, adj, qs[:1024, 0], qs[:1024, 1], hops=1, max_nodes_per_hop=100, seed=0)
torch.manual_seed(0)
mod = DGCNN(int(sub.z.max()), 30).to(dev).train()


def step():
    mod.zero_grad()
    out = mod(sub, seed=1)
    out.sum().backward()
    return out


ms, _ = median_ms(step)
print(f"DGCNN fwd+bwd, 1024 subgraphs ({sub.nodes.numel()} nodes, {sub.edge_index.shape[1]} edges), k=30: {ms:.2f} ms", flush=True)
del ptr, adj, qs, sub1
torch.cuda.empty_cache()

# ---- fb-pages-food seed 0
fb = np.load(os.path.join(ROOT, "tests", "golden", "fb_pages_food_seed0.npz"))
nf = int(fb["num_nodes"][0])
ep, en = (torch.from_numpy(fb[k].astype(np.int64)).to(dev) for k in ("edge_pos", "edge_neg"))
bg = D.BaseGraph(torch.zeros((nf, 0), device=dev), None, ep, en, torch.from_numpy(fb["num_pos"]), torch.from_numpy(fb["num_neg"]), "none")
bg.preprocess()
bg.setPosDegreeFeature()
trn, tst = D.dataset(*bg.split(0)), D.dataset(*bg.split(2))
labels = tst.y.reshape(-1)[0::2]
torch.cuda.synchronize()
t0 = time.perf_counter()
mod, losses = seal_fit(trn, 10, 32, lr=1e-3, hops=1, seed=0)
torch.cuda.synchronize()
fit_s = time.perf_counter() - t0
sc = {"seal": seal_scores(mod, tst), **{k: v for k, v in heuristic_scores(tst).items() if k in ("cn", "aa")},
      "ppr": global_heuristic_scores(tst, "ppr")}
print(f"# fb-pages-food seed 0: seal_fit {fit_s:.2f} s ({losses.numel()} steps, last loss {float(losses[-1]):.4f})")
for name, s_ in sc.items():
    rk = rank_scores(s_, tst, (20, 50, 100))
    print(f"fb-pages-food test {name}: AUC {float(ops.auc(s_, labels)[0]):.4f} " + " ".join(f"{k} {v:.4f}" for k, v in rk.items()))
print("reference (BASELINE.md): SEAL AUC 0.8661 in 35.12 s - another split, context only")
