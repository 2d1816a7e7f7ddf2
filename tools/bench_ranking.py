"""Time of the ranking-evaluation ops against a plain torch formulation of the same metric, alternating in one process:
  ops.hits_at_k              3e6 scores (2e5 positives), ks = (20, 50, 100)   vs  topk of the negatives + compare
  ops.rank_metrics           1e6 positives x 100 negatives, ks = (1, 3, 10)   vs  (neg > pos[:, None]).sum(1), (neg >= ...)
  ops.sample_tail_negatives  collab-scale R-MAT (2^18 nodes, 1.3 M edge samples), 50 000 sources x 100 negatives
CUDA-event time, median of `reps` after one warm-up; the hits_at_k inputs (24 MB) fit in L2, the rank_metrics ones (400 MB) do not.
The two formulations' results are compared too (hits exactly, MRR to 1e-12 relative).   python tools/bench_ranking.py [reps]"""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "link-prediction-gnn_b200")):
    sys.path.insert(0, p)
import torch

import bench
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


def duel(name, ours, theirs):
    """alternate the two, `reps` times each after one warm-up of both; -> (our result, their result)."""
    r0, r1 = ours(), theirs()
    t0, t1 = [], []
    for _ in range(reps):
        t, r0 = event_ms(ours)
        t0.append(t)
        t, r1 = event_ms(theirs)
        t1.append(t)
    m0, m1 = sorted(t0)[reps // 2], sorted(t1)[reps // 2]
    print(f"{name:34s} ours {m0:8.3f} ms   torch {m1:8.3f} ms   (min {min(t0):.3f} / {min(t1):.3f})", flush=True)
    return r0, r1


g = torch.Generator(device=dev).manual_seed(0)

# ---- hits@K against shared negatives
n, n_pos, ks = 3_000_000, 200_000, (20, 50, 100)
score = torch.randn(n, generator=g, device=dev)
label = torch.zeros(n, device=dev)
label[torch.randperm(n, generator=g, device=dev)[:n_pos]] = 1.0


def torch_hits():
    m = label > 0.5
    pos, neg = score[m], score[~m]
    top = torch.topk(neg, max(ks)).values
    return torch.stack([(pos > top[k - 1]).sum() for k in ks]).double() / pos.numel()


a, b = duel(f"hits_at_k  n={n}", lambda: ops.hits_at_k(score, label, ks)[:len(ks)], torch_hits)
assert torch.equal(a, b), (a, b)

# ---- MRR / hits@k against per-positive negatives
P, k, rks = 1_000_000, 100, (1, 3, 10)
pos = torch.randn(P, generator=g, device=dev)
neg = torch.randn(P, k, generator=g, device=dev)


def torch_rank():
    p = pos[:, None]
    rank = 0.5 * ((neg > p).sum(1) + (neg >= p).sum(1)).double() + 1
    return torch.cat(((1.0 / rank).mean().reshape(1), torch.stack([(rank <= kk).sum() for kk in rks]).double() / P))


a, b = duel(f"rank_metrics  {P} x {k}", lambda: ops.rank_metrics(pos, neg, rks)[:1 + len(rks)], torch_rank)
assert torch.equal(a[1:], b[1:]) and abs(float(a[0] - b[0])) <= 1e-12 * float(b[0]), (a, b)
del neg

# ---- per-source filtered negatives at collab scale
scale, samples, abcd, _ = bench.WORKLOADS["collab"]
s, d, nn = rmat_edges(scale, samples, abcd, 0, dev)
src = torch.randint(0, nn, (50_000,), generator=g, device=dev)
ts = []
out = ops.sample_tail_negatives(s, d, nn, src, 100, seed=1)
for r in range(reps):
    t, out = event_ms(lambda: ops.sample_tail_negatives(s, d, nn, src, 100, seed=2 + r))
    ts.append(t)
print(f"{'sample_tail_negatives':34s} ours {sorted(ts)[reps // 2]:8.3f} ms   (n = {nn}, {s.numel()} edges, 50000 x 100; "
      f"includes the host read of the unfilled count)", flush=True)
