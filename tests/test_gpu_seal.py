"""SEAL on the device: enclosing-subgraph extraction with DRNL labels (ops.seal_subgraphs / seal_subgraph_sizes), the DGCNN kernels
(twowl::seal_input, seal_tanh(_concat), sort_pool, bias_act, im2col), TwoWL.model.seal.DGCNN and train.seal_fit / seal_scores.

Extraction is compared exactly with a restatement of the SEAL authors' k_hop_subgraph (Python sets), the target-edge removal and
PyG's drnl_node_labeling (scipy.sparse.csgraph.shortest_path). The kernels and the whole DGCNN are compared with float64 torch on
the CPU: torch.sort(stable=True), max_pool1d, conv1d, and the oracle's GCNConv loading the same state_dict. fp32 error bound of a
compared tensor: 16 n u max|ref|, n the longest summation on its path (u = 2^-24), which covers n-term sums of terms of that size
through the tanh / ReLU / max-pool steps (each 1-Lipschitz).
"""
import numpy as np
import pytest
import scipy.sparse as sp
from scipy.sparse.csgraph import shortest_path
import torch

from test_gpu_heuristics import FAKE, EINVAL, ENOSPC, L, _err, cu, np_adjacency  # noqa: F401  (L is a fixture)
from test_gpu_recommend import fbg  # noqa: F401  (a fixture: fb-pages-food's graph and the reference model)

U32 = 2.0 ** -24
M64 = (1 << 64) - 1


# ------------------------------------------------------------------------------ CPU: argument checks

def test_seal_argument_errors(L):
    lib = L.lib
    nb = lib.twowl_seal_workspace_bytes(100, 10, 2)
    assert nb > lib.twowl_seal_workspace_bytes(100, 10, 1) > 0
    assert lib.twowl_seal_workspace_bytes(-1, 10, 1) == 0 and lib.twowl_seal_workspace_bytes(100, 10, 0) == 0
    f = lib.twowl_seal_count

    def call(n=100, Q=10, hops=1, cap=0, blocks=2, base=0, ptr=FAKE, u=FAKE, out=FAKE, ws=FAKE, wsb=nb):
        return f(ptr, FAKE, n, u, 1, FAKE, 1, Q, base, hops, cap, 7, blocks, out, FAKE, FAKE, ws, wsb, None)

    for kw in (dict(n=-1), dict(Q=-1), dict(blocks=0), dict(base=-1), dict(base=1 << 31)):
        _err(L, call(**kw), EINVAL, "bad sizes")
    for h in (0, 4, -1):
        _err(L, call(hops=h), EINVAL, "hops must be")
    _err(L, call(cap=-1), EINVAL, "max_nodes_per_hop")
    for kw in ("ptr", "u", "out", "ws"):
        _err(L, call(**{kw: None}), EINVAL, "null pointer")
    _err(L, call(wsb=nb - 1), ENOSPC, "workspace too small")
    g = lib.twowl_seal_fill
    _err(L, g(FAKE, FAKE, 100, FAKE, 1, FAKE, 1, 10, 0, 2, 0, 7, 2, FAKE, FAKE, -1, FAKE, FAKE, FAKE, FAKE, nb, None), EINVAL, "bad sizes")
    _err(L, g(FAKE, FAKE, 100, FAKE, 1, FAKE, 1, 10, 0, 2, 0, 7, 2, FAKE, FAKE, 5, None, FAKE, FAKE, FAKE, nb, None), EINVAL,
         "null pointer")
    _err(L, g(FAKE, FAKE, 100, FAKE, 1, FAKE, 1, 10, 0, 2, 0, 7, 2, FAKE, FAKE, 5, FAKE, FAKE, None, FAKE, nb, None), EINVAL,
         "null pointer")


def test_dgcnn_kernel_argument_errors(L):
    lib = L.lib
    _err(L, lib.twowl_label_gather(FAKE, 0, 5, FAKE, 3, 0, FAKE, None), EINVAL, "bad sizes")
    _err(L, lib.twowl_label_gather(None, 4, 5, FAKE, 3, 0, FAKE, None), EINVAL, "null pointer")
    _err(L, lib.twowl_tanh_slice_fwd(FAKE, 3, 4, FAKE, 4, 1, None), EINVAL, "bad sizes")
    _err(L, lib.twowl_tanh_slice_fwd(None, 3, 4, FAKE, 8, 1, None), EINVAL, "null pointer")
    _err(L, lib.twowl_tanh_slice_bwd(FAKE, FAKE, 8, -1, 3, 4, FAKE, None), EINVAL, "bad sizes")
    _err(L, lib.twowl_tanh_slice_bwd(FAKE, None, 8, 0, 3, 4, FAKE, None), EINVAL, "null pointer")
    _err(L, lib.twowl_sortpool_fwd(FAKE, 8, 8, FAKE, 2, 10, FAKE, FAKE, None), EINVAL, "bad sizes")
    _err(L, lib.twowl_sortpool_fwd(FAKE, 8, 7, FAKE, 2, 0, FAKE, FAKE, None), EINVAL, "bad sizes")
    _err(L, lib.twowl_sortpool_fwd(FAKE, 8, 7, None, 2, 10, FAKE, FAKE, None), EINVAL, "null pointer")
    _err(L, lib.twowl_sortpool_bwd(FAKE, None, 2, 10, 8, 5, FAKE, None), EINVAL, "null pointer")
    for pool in (0, 3):
        _err(L, lib.twowl_bias_act_fwd(FAKE, FAKE, 2, 10, 16, pool, 1, 0.0, 0, FAKE, None), EINVAL, "bad sizes")
    _err(L, lib.twowl_bias_act_fwd(FAKE, FAKE, 2, 10, 16, 1, 1, 1.0, 0, FAKE, None), EINVAL, "p_drop")
    _err(L, lib.twowl_bias_act_bwd(FAKE, FAKE, None, 2, 10, 16, 1, 1, 0.0, 0, FAKE, None), EINVAL, "null pointer")
    _err(L, lib.twowl_im2col_fwd(FAKE, 2, 4, 16, 5, FAKE, None), EINVAL, "bad sizes")
    _err(L, lib.twowl_im2col_bwd(None, 2, 5, 16, 5, FAKE, None), EINVAL, "null pointer")


def test_seal_ops_refuse_cpu_tensors(L):
    from twowl_b200 import ops
    ptr, adj, s = torch.zeros(6, dtype=torch.int64), torch.zeros(0, dtype=torch.int32), torch.zeros(3, dtype=torch.int64)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.seal_subgraphs(ptr, adj, s, s + 1)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.seal_subgraph_sizes(ptr, adj, s, s + 1)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.sortpool_fwd(torch.zeros((4, 8)), s, 10, 7)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.label_gather(torch.zeros((4, 8)), s)


# ------------------------------------------------------------------------------ restatements

def hash_u32(seed, idx):
    z = (idx + seed * 0x9E3779B97F4A7C15 + 0x9E3779B97F4A7C15) & M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M64
    return (z ^ (z >> 31)) >> 32


def ref_subgraph(hp, ha, u, v, hops, cap, seed, qidx):
    """The SEAL authors' k_hop_subgraph with the cap rule, target-edge removal and PyG's drnl_node_labeling -> (nodes, rows, cols, z)."""
    nodes, seen, fringe = [u, v], {u, v}, {u, v}
    for _ in range(hops):
        cand = set()
        for x in fringe:
            cand.update(ha[hp[x]:hp[x + 1]].tolist())
        cand -= seen
        seen |= cand
        if cap and len(cand) > cap:
            cand = sorted(cand, key=lambda y: (hash_u32(seed, (qidx << 32) | y), y))[:cap]
        fringe = set(cand)
        nodes += list(cand)
    nodes = np.array(sorted(nodes), np.int64)
    n = nodes.size
    pos = {x: i for i, x in enumerate(nodes.tolist())}
    rows, cols = [], []
    for i, x in enumerate(nodes.tolist()):
        for y in ha[hp[x]:hp[x + 1]].tolist():
            if y in pos and not ((x == u and y == v) or (x == v and y == u)):
                rows.append(i), cols.append(pos[y])
    adj = sp.csr_matrix((np.ones(len(rows)), (rows, cols)), shape=(n, n))
    src, dst = sorted((pos[u], pos[v]))
    idx = list(range(src)) + list(range(src + 1, n))
    adj_wo_src = adj[idx, :][:, idx]
    idx = list(range(dst)) + list(range(dst + 1, n))
    adj_wo_dst = adj[idx, :][:, idx]
    d2s = np.insert(shortest_path(adj_wo_dst, directed=False, unweighted=True, indices=src), dst, 0, axis=0)
    d2d = np.insert(shortest_path(adj_wo_src, directed=False, unweighted=True, indices=dst - 1), src, 0, axis=0)
    d2s, d2d = torch.from_numpy(d2s), torch.from_numpy(d2d)
    dist = d2s + d2d
    h, m = dist // 2, dist % 2
    z = 1 + torch.min(d2s, d2d)
    z += h * (h + m - 1)
    z[src] = 1.
    z[dst] = 1.
    z[torch.isnan(z)] = 0.
    return nodes, np.array(rows, np.int64), np.array(cols, np.int64), z.to(torch.long).numpy()


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from twowl_b200 import ops as o
    return o


def _rmat(n_log, m, rng):
    a, b, c = 0.57, 0.19, 0.19
    r = np.zeros(m, np.int64)
    col = np.zeros(m, np.int64)
    for _ in range(n_log):
        x = rng.random(m)
        r = 2 * r + (x > a + b)
        col = 2 * col + (((x > a) & (x <= a + b)) | (x > a + b + c))
    return r, col


def _graphs():
    rng = np.random.default_rng(5)
    n = 400
    er = (rng.integers(0, 300, 900), rng.integers(0, 300, 900), n)                  # 300..399 isolated
    rr, rc = _rmat(10, 6000, rng)
    rmat = (rr, rc, 1024)
    hub_r = np.concatenate([np.zeros(3000, np.int64), rng.integers(1, 3200, 4000)])
    hub_c = np.concatenate([np.arange(1, 3001), rng.integers(1, 3200, 4000)])
    hub = (hub_r, hub_c, 3300)                                                         # 3200..3299 isolated
    return {"er": er, "rmat": rmat, "hub": hub}


def _queries(hp, ha, n, rng):
    deg = np.diff(hp)
    iso = np.flatnonzero(deg == 0)
    e = rng.integers(0, ha.size, 12)
    rows = np.searchsorted(hp, e, side="right") - 1
    pos = np.stack([rows, ha[e]], 1)                                                   # edges present
    neg = rng.integers(0, n, (12, 2))
    neg = neg[neg[:, 0] != neg[:, 1]]
    act = np.flatnonzero(deg > 0)
    extra = [[iso[0], act[0]], [iso[0], iso[1]], [act[1], iso[-1]], [int(np.argmax(deg)), act[2]]]
    q = np.concatenate([pos, neg, np.array(extra, np.int64)])
    q = np.concatenate([q, q[:3]])                                                       # duplicated queries
    return q[q[:, 0] != q[:, 1]]


def _check_batch(sub, hp, ha, q, hops, cap, seed, base=0):
    node_ptr = sub.node_ptr.cpu().numpy()
    nodes, z, ei = sub.nodes.cpu().numpy(), sub.z.cpu().numpy(), sub.edge_index.cpu().numpy()
    assert np.array_equal(sub.batch.cpu().numpy(), np.repeat(np.arange(len(q)), np.diff(node_ptr)))
    e0 = 0
    for i, (u, v) in enumerate(q.tolist()):
        rn, rr, rcol, rz = ref_subgraph(hp, ha, u, v, hops, cap, seed, base + i)
        a, b = node_ptr[i], node_ptr[i + 1]
        assert np.array_equal(nodes[a:b], rn), (i, u, v)
        assert np.array_equal(z[a:b], rz), (i, u, v, z[a:b], rz)
        m = rr.size
        assert np.array_equal(ei[0, e0:e0 + m], rr + a) and np.array_equal(ei[1, e0:e0 + m], rcol + a), (i, u, v)
        e0 += m
    assert e0 == ei.shape[1]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["er", "rmat", "hub"])
def test_subgraphs_match_restatement(ops, name):
    r, c, n = _graphs()[name]
    ptr, adj = ops.simple_adjacency(cu(r), cu(c), n)
    hp, ha = ptr.cpu().numpy(), adj.cpu().numpy()
    q = _queries(hp, ha, n, np.random.default_rng(11))
    for hops in (1, 2, 3):
        for cap in (0, 7, 40):
            sub = ops.seal_subgraphs(ptr, adj, cu(q[:, 0]), cu(q[:, 1]), hops=hops, max_nodes_per_hop=cap, seed=3)
            _check_batch(sub, hp, ha, q, hops, cap, 3)
            sizes = ops.seal_subgraph_sizes(ptr, adj, cu(q[:, 0]), cu(q[:, 1]), hops=hops, max_nodes_per_hop=cap, seed=3)
            assert torch.equal(sizes, sub.node_ptr[1:] - sub.node_ptr[:-1])


@pytest.mark.gpu
def test_subgraphs_batching_repeatability_and_errors(ops):
    r, c, n = _graphs()["hub"]
    ptr, adj = ops.simple_adjacency(cu(r), cu(c), n)
    q = _queries(ptr.cpu().numpy(), adj.cpu().numpy(), n, np.random.default_rng(2))
    u, v = cu(q[:, 0]), cu(q[:, 1])
    kw = dict(hops=2, max_nodes_per_hop=50, seed=9)
    ref = ops.seal_subgraphs(ptr, adj, u, v, **kw)
    fields = ("node_ptr", "nodes", "z", "edge_index")
    for ws in (None, 1, 3 * 20 * n):                 # one CTA at a time, three, the default
        got = ops.seal_subgraphs(ptr, adj, u, v, max_workspace=ws, **kw)
        assert all(torch.equal(getattr(got, f), getattr(ref, f)) for f in fields)
    # cut in two calls with index_base: the same subgraphs
    h = len(q) // 2
    a = ops.seal_subgraphs(ptr, adj, u[:h], v[:h], **kw)
    b = ops.seal_subgraphs(ptr, adj, u[h:], v[h:], index_base=h, **kw)
    na = a.nodes.numel()
    assert torch.equal(torch.cat((a.nodes, b.nodes)), ref.nodes) and torch.equal(torch.cat((a.z, b.z)), ref.z)
    assert torch.equal(torch.cat((a.edge_index, b.edge_index + na), 1), ref.edge_index)
    # the uncapped 1-hop subgraph of the degree-3000 hub
    big = ops.seal_subgraphs(ptr, adj, cu([0]), cu([5]), hops=1)
    _check_batch(big, ptr.cpu().numpy(), adj.cpu().numpy(), np.array([[0, 5]]), 1, 0, 0)
    assert big.nodes.numel() > 3000
    empty = ops.seal_subgraphs(ptr, adj, u[:0], v[:0])
    assert empty.node_ptr.tolist() == [0] and empty.nodes.numel() == 0 and empty.edge_index.shape == (2, 0)
    with pytest.raises(IndexError):
        ops.seal_subgraphs(ptr, adj, cu([0, n]), cu([1, 2]))
    with pytest.raises(IndexError):
        ops.seal_subgraphs(ptr, adj, cu([-1]), cu([1]))
    with pytest.raises(ValueError, match="u == v"):
        ops.seal_subgraphs(ptr, adj, cu([3, 4]), cu([3, 5]))
    with pytest.raises(ValueError, match="hops"):
        ops.seal_subgraphs(ptr, adj, u, v, hops=4)


# ------------------------------------------------------------------------------ DGCNN kernels against float64 torch

def _bound(ref, n):
    return 16 * n * U32 * float(ref.abs().max()) + 1e-30


def _close(got, ref, n, what):
    got = got.detach().cpu().double()
    err = float((got - ref).abs().max()) if ref.numel() else 0.0
    assert err <= _bound(ref, n), (what, err, _bound(ref, n))


@pytest.mark.gpu
def test_sortpool_against_torch(ops):
    from twowl_b200 import functional as F2
    rng = np.random.default_rng(0)
    sizes = [1, 10, 4, 25, 10, 3]                   # one row, exactly k, fewer than k, more than k
    k, D = 10, 12
    n = sum(sizes)
    X = torch.from_numpy(rng.standard_normal((n, D)).astype(np.float32))
    X[3:7, D - 1] = 0.25                            # exact ties in the key column
    X[20:30, D - 1] = -1.0
    gptr = torch.tensor(np.concatenate([[0], np.cumsum(sizes)]), dtype=torch.int64)
    Xd = X.cuda().requires_grad_()
    out, idx = F2.sort_pool(Xd, gptr.cuda(), k, D - 1)
    G = torch.from_numpy(rng.standard_normal((len(sizes), k, D)).astype(np.float32))
    out.backward(G.cuda())
    X64 = X.double().requires_grad_()
    ref = torch.zeros((len(sizes), k, D), dtype=torch.float64)
    rows = []
    for b in range(len(sizes)):
        blk = X64[gptr[b]:gptr[b + 1]]
        order = torch.sort(blk[:, -1], descending=True, stable=True).indices[:k]
        ref[b, :order.numel()] = blk[order]
        rows.append(order + gptr[b])
    ref.backward(G.double())
    assert torch.equal(out.detach().cpu().double(), ref.detach())
    assert torch.equal(Xd.grad.cpu().double(), X64.grad)
    exp_idx = torch.full((len(sizes), k), -1, dtype=torch.int32)
    for b, r in enumerate(rows):
        exp_idx[b, :r.numel()] = r.to(torch.int32)
    assert torch.equal(idx.cpu(), exp_idx)


@pytest.mark.gpu
def test_conv_head_pieces_against_torch(ops):
    from twowl_b200 import functional as F2
    rng = np.random.default_rng(1)
    B, k, C = 5, 11, 16                             # odd k: the last row is dropped by MaxPool1d(2, 2)
    Y = rng.standard_normal((B * k, C)).astype(np.float32)
    Y[0:2, 3] = 0.5                                 # an exact tie inside a pooling window
    bias = rng.standard_normal(C).astype(np.float32)
    Yd, bd = torch.from_numpy(Y).cuda().requires_grad_(), torch.from_numpy(bias).cuda().requires_grad_()
    P = F2.bias_act(Yd, bd, B, 2, True, 0.0, 0)
    Xc = F2.im2col(P, B, 5)
    W2 = rng.standard_normal((32, C, 5)).astype(np.float32)
    out = F2.linear(Xc, torch.from_numpy(W2).reshape(32, C * 5).cuda())
    Gout = rng.standard_normal(out.shape).astype(np.float32)
    out.backward(torch.from_numpy(Gout).cuda())
    # float64 torch: [B, C, k] layout
    Y64 = torch.from_numpy(Y).double().reshape(B, k, C).transpose(1, 2).requires_grad_()
    b64 = torch.from_numpy(bias).double().requires_grad_()
    P64 = torch.nn.functional.max_pool1d(torch.relu(Y64 + b64.view(1, C, 1)), 2, 2)
    o64 = torch.nn.functional.conv1d(P64, torch.from_numpy(W2).double())          # [B, 32, L2]
    o64.backward(torch.from_numpy(Gout).double().reshape(B, -1, 32).transpose(1, 2))
    _close(P, P64.detach().transpose(1, 2).reshape(-1, C), 1, "pool")
    _close(out, o64.detach().transpose(1, 2).reshape(-1, 32), C * 5, "conv2")
    _close(Yd.grad, Y64.grad.transpose(1, 2).reshape(-1, C), 32 * 5, "dY")
    _close(bd.grad, b64.grad, B * k * 32 * 5, "dbias")


# ------------------------------------------------------------------------------ the whole DGCNN against a float64 restatement

class RefDGCNN(torch.nn.Module):
    def __init__(self, mod):
        super().__init__()
        from oracle.pyg_shim.torch_geometric.nn import GCNConv
        self.convs = torch.nn.ModuleList([GCNConv(c.in_channels, c.out_channels) for c in mod.convs])
        self.conv1 = torch.nn.Conv1d(1, 16, mod.D, mod.D)
        self.conv2 = torch.nn.Conv1d(16, 32, 5, 1)
        self.mlp = torch.nn.Module()
        self.mlp.lins = torch.nn.ModuleList([torch.nn.Linear(32 * mod.L2, 128), torch.nn.Linear(128, 1)])
        self.k = mod.k
        self.load_state_dict({k_: v.detach().cpu() for k_, v in mod.state_dict().items()})
        self.double()

    def forward(self, x, ei, node_ptr):
        xs = [x]
        for conv in self.convs:
            xs.append(conv(xs[-1], ei).tanh())
        X = torch.cat(xs[1:], -1)
        B = node_ptr.numel() - 1
        S = X.new_zeros((B, self.k, X.shape[1]))
        for b in range(B):
            blk = X[node_ptr[b]:node_ptr[b + 1]]
            order = torch.sort(blk[:, -1], descending=True, stable=True).indices[:self.k]
            S[b, :order.numel()] = blk[order]
        h = torch.relu(self.conv1(S.reshape(B, 1, -1)))
        h = torch.nn.functional.max_pool1d(h, 2, 2)
        h = torch.relu(self.conv2(h)).reshape(B, -1)
        h = torch.relu(self.mlp.lins[0](h))
        return self.mlp.lins[1](h)


def _small_batch(ops, n_q=24, hops=2):
    r, c, n = _graphs()["er"]
    ptr, adj = ops.simple_adjacency(cu(r), cu(c), n)
    q = _queries(ptr.cpu().numpy(), adj.cpu().numpy(), n, np.random.default_rng(4))[:n_q]
    return ops.seal_subgraphs(ptr, adj, cu(q[:, 0]), cu(q[:, 1]), hops=hops, max_nodes_per_hop=15, seed=1), n


@pytest.mark.gpu
@pytest.mark.parametrize("F", [0, 6])
def test_dgcnn_against_float64_restatement(ops, F):
    from TwoWL.model.seal import DGCNN
    sub, n = _small_batch(ops)
    torch.manual_seed(0)
    max_z = int(sub.z.max())
    mod = DGCNN(max_z, 12, hidden=32, num_layers=3, node_feat_dim=F).cuda().train()
    mod.dropout = 0.0
    feat = torch.randn((n, F)).cuda() if F else None
    w = torch.randn((sub.num_graphs, 1))
    out = mod(sub, feat)
    (out * w.cuda()).sum().backward()
    ref = RefDGCNN(mod)
    x = torch.nn.functional.one_hot(sub.z.cpu().to(torch.int64), max_z + 1).double()
    if F:
        x = torch.cat((x, feat.cpu().double()[sub.nodes.cpu()]), 1)
    o64 = ref(x, sub.edge_index.cpu(), sub.node_ptr.cpu())
    (o64 * w.double()).sum().backward()
    deg = int(torch.bincount(sub.edge_index[1].cpu(), minlength=sub.nodes.numel()).max()) + 1
    nt = max(mod.Dp, 32 * mod.L2, 128, deg * (max_z + 1 + F), mod.k * 16)
    _close(out, o64.detach(), nt, "logits")
    grads = dict(ref.named_parameters())
    for name, p in mod.named_parameters():
        _close(p.grad, grads[name].grad, nt * sub.nodes.numel(), f"grad {name}")


@pytest.mark.gpu
def test_dgcnn_dropout_repeatable(ops):
    from TwoWL.model.seal import DGCNN
    sub, n = _small_batch(ops)
    torch.manual_seed(0)
    mod = DGCNN(int(sub.z.max()), 10).cuda().train()
    res = []
    for _ in range(2):
        mod.zero_grad()
        out = mod(sub, seed=12345)
        out.sum().backward()
        res.append([out.detach().clone()] + [p.grad.clone() for p in mod.parameters()])
    assert all(torch.equal(a, b) for a, b in zip(*res))
    mod.zero_grad()
    other = mod(sub, seed=777)
    assert not torch.equal(other.detach(), res[0][0])


# ------------------------------------------------------------------------------ training

@pytest.mark.gpu
def test_seal_fit_repeatable(fbg):
    from TwoWL.model.train import seal_fit
    D, bg, _ = fbg
    trn = D.dataset(*bg.split(0))
    runs = [seal_fit(trn, 1, 64, lr=1e-3, max_nodes_per_hop=20, seed=4) for _ in range(2)]
    (m0, l0), (m1, l1) = runs
    assert torch.equal(l0, l1) and l0.numel() > 0 and bool(torch.isfinite(l0).all())
    for (k0, a), (k1, b) in zip(m0.state_dict().items(), m1.state_dict().items()):
        assert k0 == k1 and torch.equal(a, b), k0


# measured on one B200 (1000 W power limit) with these settings: test AUC 0.925 (CN 0.845, AA 0.847, PPR 0.880, node2vec 0.856);
# the floor sits 0.045 below it
SEAL_FB = dict(epochs=10, batch_size=32, lr=1e-3, hops=1, seed=0)
AUC_FLOOR = 0.88


@pytest.mark.gpu
def test_seal_end_to_end_fb_pages_food(fbg):
    import time
    from TwoWL.model.train import embedding_scores, global_heuristic_scores, heuristic_scores, node2vec_embedding, rank_scores, \
        seal_fit, seal_scores
    from twowl_b200 import ops
    D, bg, _ = fbg
    trn, tst = D.dataset(*bg.split(0)), D.dataset(*bg.split(2))
    t0 = time.perf_counter()
    mod, losses = seal_fit(trn, **SEAL_FB)
    torch.cuda.synchronize()
    secs = time.perf_counter() - t0
    s = seal_scores(mod, tst, hops=SEAL_FB["hops"])
    P = tst.y.shape[0] // 2
    assert s.shape == (P,) and s.dtype == torch.float32 and bool(torch.isfinite(s).all())
    assert torch.equal(s, seal_scores(mod, tst, hops=SEAL_FB["hops"], batch_size=37))
    labels = tst.y.reshape(-1)[0::2]
    ks = (20, 50, 100)
    rows = {"seal": s, **{k: v for k, v in heuristic_scores(tst).items() if k in ("cn", "aa")},
            "ppr": global_heuristic_scores(tst, "ppr"), "node2vec": embedding_scores(tst, node2vec_embedding(tst, epochs=20, batch_walks=128)[0])}
    table = {name: (float(ops.auc(sc, labels)[0]), rank_scores(sc, tst, ks)) for name, sc in rows.items()}
    for name, (auc, rk) in table.items():
        print(f"fb-pages-food test {name}: AUC {auc:.4f} " + " ".join(f"{k} {v:.4f}" for k, v in rk.items()))
    print(f"SEAL training {secs:.2f} s, {losses.numel()} steps, last loss {float(losses[-1]):.4f}")
    assert losses[-1] < losses[0]
    assert table["seal"][0] > AUC_FLOOR, table["seal"][0]
