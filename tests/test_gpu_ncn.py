"""Neural Common Neighbor on the device: the common-neighbour lists (twowl_common_neighbors_count / _fill, ops.common_neighbors), the
adjacency pair mask (twowl_adjacency_pair_mask), twowl::cn_aggregate, TwoWL.model.ncn.NCN and train.ncn_fit / ncn_scores /
rerank_scores.

The lists are compared exactly with np.intersect1d of the two neighbour lists, over the graph with the masked edges deleted by
scipy.sparse. cn_aggregate and the whole NCN are compared with float64 torch on the CPU (the oracle's gcn_conv on the graph without
the batch's positive edges, scipy common neighbours, torch MLPs loading the same state_dict). cn_aggregate is held to the
fp32 bound of test_gpu_seal.py, 16 n u max|ref| with n the longest summation; the whole NCN's logits and gradients within 1e-4 of
float64 in norm per tensor, a bound the test shows that halved, zeroed or incomplete gradients break.
"""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

from test_gpu_heuristics import FAKE, EINVAL, ENOSPC, L, _err, _queries, cu, np_adjacency  # noqa: F401  (L is a fixture)
from test_gpu_recommend import fbg  # noqa: F401  (a fixture: fb-pages-food's graph and the reference model)
from test_gpu_seal import _close, _rmat

# ------------------------------------------------------------------------------ CPU: argument checks


def test_common_neighbors_argument_errors(L):
    lib = L.lib
    nb = lib.twowl_common_neighbors_count_workspace_bytes(1000, 100)
    assert nb >= lib.twowl_common_neighbors_count_workspace_bytes(0, 0) > 0
    f = lib.twowl_common_neighbors_count

    def count(n=50, P=1000, nch=100, ptr=FAKE, u=FAKE, cp=FAKE, cb=FAKE, off=FAKE, wsb=nb):
        return f(ptr, FAKE, n, None, u, 1, FAKE, 1, P, off, nch, cp, cb, FAKE, wsb, None)

    for kw in (dict(P=-1), dict(P=1 << 31), dict(n=-1), dict(n=(1 << 31) - 1), dict(nch=-1)):
        _err(L, count(**kw), EINVAL, "bad sizes")
    for kw in ("ptr", "u", "cp", "cb", "off"):
        _err(L, count(**{kw: None}), EINVAL, "null pointer")
    _err(L, count(wsb=nb - 1), ENOSPC, "workspace too small")
    g = lib.twowl_common_neighbors_fill

    def fill(n=50, P=1000, nch=100, nnz=10, ptr=FAKE, adj=FAKE, ids=FAKE, pair=FAKE, cp=FAKE):
        return g(ptr, adj, n, None, FAKE, 1, FAKE, 1, P, FAKE, nch, cp, FAKE, nnz, ids, pair, None)

    for kw in (dict(P=-1), dict(n=-1), dict(nch=-1), dict(nnz=-1), dict(nnz=1 << 31)):
        _err(L, fill(**kw), EINVAL, "bad sizes")
    for kw in ("ptr", "adj", "ids", "pair", "cp"):
        _err(L, fill(**{kw: None}), EINVAL, "null pointer")
    h = lib.twowl_adjacency_pair_mask
    _err(L, h(FAKE, FAKE, 50, 100, FAKE, 1, FAKE, 1, -1, FAKE, FAKE, None), EINVAL, "bad sizes")
    _err(L, h(FAKE, FAKE, -1, 100, FAKE, 1, FAKE, 1, 10, FAKE, FAKE, None), EINVAL, "bad sizes")
    _err(L, h(FAKE, FAKE, 50, -1, FAKE, 1, FAKE, 1, 10, FAKE, FAKE, None), EINVAL, "bad sizes")
    _err(L, h(FAKE, FAKE, 50, 100, FAKE, 1, FAKE, 1, 10, None, FAKE, None), EINVAL, "null pointer")
    _err(L, h(FAKE, FAKE, 50, 100, FAKE, 1, FAKE, 1, 10, FAKE, None, None), EINVAL, "null pointer")
    _err(L, h(FAKE, FAKE, 50, 100, None, 1, FAKE, 1, 10, FAKE, FAKE, None), EINVAL, "null pointer")


def test_ncn_ops_refuse_cpu_tensors(L):
    from twowl_b200 import ops
    ptr, adj, s = torch.zeros(6, dtype=torch.int64), torch.zeros(0, dtype=torch.int32), torch.zeros(3, dtype=torch.int64)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.common_neighbors(ptr, adj, s, s + 1)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.adjacency_pair_mask(ptr, adj, s, s + 1)


def test_ncn_parameter_names(L):
    from TwoWL.model.ncn import NCN
    keys = set(NCN(7, hidden=16, num_layers=3).state_dict())
    assert keys == {"emb.weight", "lin_ij.weight", "lin_ij.bias", "lin_cn.weight", "lin_cn.bias", "lin_h.weight", "lin_h.bias",
                    "lin_o.weight", "lin_o.bias"} | {f"convs.{i}.{p}" for i in range(3) for p in ("lin.weight", "bias")}
    m = NCN(7, hidden=16, cn=False, node_feat_dim=6)
    assert "emb.weight" not in m.state_dict() and "lin_cn.weight" not in m.state_dict()
    assert m.convs[0].lin.weight.shape == (16, 6) and m.lin_h.weight.shape == (16, 16)
    with pytest.raises(ValueError, match="multiple of 4"):
        NCN(7, hidden=10)


# ------------------------------------------------------------------------------ restatements

def np_lists(hp, ha, u, v, mask=None):
    """CN of every pair (np.intersect1d over the unmasked entries) -> (ptr, ids, pair)."""
    keep = np.ones(ha.size, bool) if mask is None else mask == 0
    rows = [np.intersect1d(ha[hp[a]:hp[a + 1]][keep[hp[a]:hp[a + 1]]], ha[hp[b]:hp[b + 1]][keep[hp[b]:hp[b + 1]]])
            for a, b in zip(u.tolist(), v.tolist())]
    lens = np.array([r.size for r in rows], np.int64)
    ids = np.concatenate(rows).astype(np.int32) if rows else np.zeros(0, np.int32)
    return np.concatenate([[0], np.cumsum(lens)]), ids, np.repeat(np.arange(len(rows)), lens).astype(np.int32)


def deleted_graph(hp, ha, pairs):
    """(ptr, adj) of the simple graph without the edges {a, b} of `pairs` (scipy.sparse)."""
    n = hp.size - 1
    A = sp.csr_matrix((np.ones(ha.size), ha.astype(np.int64), hp), shape=(n, n)).tolil()
    for a, b in pairs.tolist():
        if a != b:
            A[a, b] = 0
            A[b, a] = 0
    A = A.tocsr()
    A.eliminate_zeros()
    A.sort_indices()
    return A.indptr.astype(np.int64), A.indices.astype(np.int32)


def check_lists(cn, ref, what):
    rp, ri, rq = ref
    assert np.array_equal(cn.ptr.cpu().numpy(), rp), f"{what}: counts differ"
    assert np.array_equal(cn.ids.cpu().numpy(), ri), f"{what}: ids differ"
    assert np.array_equal(cn.pair.cpu().numpy(), rq), f"{what}: pair index differs"


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from twowl_b200 import ops as o
    return o


def _graphs():
    rng = np.random.default_rng(7)
    er = (rng.integers(0, 300, 1500), rng.integers(0, 300, 1500), 400)                 # 300..399 isolated
    rr, rc = _rmat(10, 8000, rng)
    # two hubs sharing 1500 neighbours (every pair of them takes the chunked path), plus noise
    hub_r = np.concatenate([np.zeros(2500, np.int64), np.ones(2500, np.int64), rng.integers(2, 4000, 3000)])
    hub_c = np.concatenate([np.arange(2, 2502), np.arange(1002, 3502), rng.integers(2, 4000, 3000)])
    return {"er": er, "rmat": (rr, rc, 1024), "hubs": (hub_r, hub_c, 4100)}


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["er", "rmat", "hubs"])
def test_common_neighbors_match_intersect1d(ops, name):
    r, c, n = _graphs()[name]
    ptr, adj = ops.simple_adjacency(cu(r), cu(c), n)
    hp, ha = ptr.cpu().numpy(), adj.cpu().numpy()
    u, v = _queries(np.random.default_rng(3), n, hp, 600)
    u, v = np.concatenate([u, [0, 1, 0, 0]]), np.concatenate([v, [1, 0, 0, 2]])       # hub pairs both ways, a hub with itself
    cn = ops.common_neighbors(ptr, adj, cu(u), cu(v))
    ref = np_lists(hp, ha, u, v)
    check_lists(cn, ref, name)
    assert torch.equal(cn.ptr.diff().float(), ops.link_heuristics(ptr, adj, cu(u), cu(v))[0])
    if name == "hubs":
        assert int(cn.ptr.diff()[-4]) == 1500                # (0, 1): chunks of a long pair, in chunk order
    again = ops.common_neighbors(ptr, adj, cu(u), cu(v))
    assert all(torch.equal(getattr(cn, f), getattr(again, f)) for f in ("ptr", "ids", "pair"))


@pytest.mark.gpu
def test_common_neighbors_edge_cases(ops):
    r, c, n = _graphs()["er"]
    ptr, adj = ops.simple_adjacency(cu(r), cu(c), n)
    empty = ops.common_neighbors(ptr, adj, cu([]), cu([]))
    assert empty.ptr.tolist() == [0] and empty.ids.numel() == 0 and empty.num_pairs == 0
    iso = ops.common_neighbors(ptr, adj, cu([350, 350, 5]), cu([360, 5, 350]))          # isolated endpoints
    assert iso.ptr.tolist() == [0, 0, 0, 0]
    p0, a0 = ops.simple_adjacency(cu([]), cu([]), 9)                                    # no edges at all
    none = ops.common_neighbors(p0, a0, cu([0, 3, 8]), cu([0, 5, 8]))
    assert none.ptr.tolist() == [0, 0, 0, 0] and none.ids.numel() == 0
    assert ops.adjacency_pair_mask(p0, a0, cu([0]), cu([3])).numel() == 0
    for bu, bv in (([0, n], [1, 2]), ([-1], [1]), ([1], [n + 5])):
        with pytest.raises(IndexError):
            ops.common_neighbors(ptr, adj, cu(bu), cu(bv))
        with pytest.raises(IndexError):
            ops.adjacency_pair_mask(ptr, adj, cu(bu), cu(bv))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["rmat", "hubs"])
def test_masked_common_neighbors_match_deleted_graph(ops, name):
    r, c, n = _graphs()[name]
    ptr, adj = ops.simple_adjacency(cu(r), cu(c), n)
    hp, ha = ptr.cpu().numpy(), adj.cpu().numpy()
    rng = np.random.default_rng(9)
    e = rng.integers(0, ha.size, 300)
    rows = np.searchsorted(hp, e, side="right") - 1
    edges = np.stack([rows, ha[e]], 1)                                                   # edges, both orientations below
    edges[::2] = edges[::2, ::-1]
    dele = np.concatenate([edges, edges[:20], rng.integers(0, n, (40, 2)), [[3, 3], [0, 1], [1, 2]]])   # duplicates, non-edges, u == v
    mask = ops.adjacency_pair_mask(ptr, adj, cu(dele[:, 0]), cu(dele[:, 1]))
    dp, da = deleted_graph(hp, ha, dele)
    # the mask marks exactly the entries the deletion removes
    kept = np.zeros(ha.size, bool)
    for x in range(n):
        kept[hp[x]:hp[x + 1]] = np.isin(ha[hp[x]:hp[x + 1]], da[dp[x]:dp[x + 1]])
    assert mask.dtype == torch.uint8 and np.array_equal(mask.cpu().numpy() == 0, kept)
    u, v = _queries(np.random.default_rng(4), n, hp, 500)
    u, v = np.concatenate([u, dele[:100, 0], dele[:100, 1], [0, 1]]), np.concatenate([v, dele[:100, 1], dele[:100, 0], [1, 1]])
    cn = ops.common_neighbors(ptr, adj, cu(u), cu(v), mask)
    check_lists(cn, np_lists(dp, da, u, v), f"{name} masked")
    again = ops.common_neighbors(ptr, adj, cu(u), cu(v), ops.adjacency_pair_mask(ptr, adj, cu(dele[:, 0]), cu(dele[:, 1])))
    assert all(torch.equal(getattr(cn, f), getattr(again, f)) for f in ("ptr", "ids", "pair"))


# ------------------------------------------------------------------------------ cn_aggregate

@pytest.mark.gpu
def test_cn_aggregate_against_float64(ops):
    from twowl_b200 import functional as F2
    r, c, n = _graphs()["hubs"]
    ptr, adj = ops.simple_adjacency(cu(r), cu(c), n)
    hp = ptr.cpu().numpy()
    u, v = _queries(np.random.default_rng(5), n, hp, 800)
    u, v = np.concatenate([u, [0, 1]]), np.concatenate([v, [1, 0]])
    cn = ops.common_neighbors(ptr, adj, cu(u), cu(v))
    rng = np.random.default_rng(6)
    h = torch.from_numpy(rng.standard_normal((n, 16)).astype(np.float32))
    G = torch.from_numpy(rng.standard_normal((len(u), 16)).astype(np.float32))
    res = []
    for _ in range(2):
        hd = h.cuda().requires_grad_()
        out = F2.cn_aggregate(hd, cn)
        out.backward(G.cuda())
        res.append((out.detach(), hd.grad))
    assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][1], res[1][1])
    ids, pair = cn.ids.cpu().long(), cn.pair.cpu().long()
    ref = torch.zeros((len(u), 16), dtype=torch.float64).index_add_(0, pair, h.double()[ids])
    dref = torch.zeros((n, 16), dtype=torch.float64).index_add_(0, ids, G.double()[pair])
    _close(res[0][0], ref, int(cn.ptr.diff().max()), "cn_aggregate")
    _close(res[0][1], dref, int(torch.bincount(ids, minlength=n).max()), "cn_aggregate backward")


# ------------------------------------------------------------------------------ NCN against a float64 restatement

def _ncn_batch(ops):
    """A doubled edge tensor (columns 2k, 2k + 1 = both directions of pair k), a batch of positives and negatives, and what
    ncn_fit hands the model for it."""
    from TwoWL.utils import double, sample_block
    r, c, n = _graphs()["rmat"]
    hp, ha = np_adjacency(r, c, n)
    rows = np.repeat(np.arange(n), np.diff(hp))
    und = np.stack([rows, ha], 1)[rows < ha]
    ei = cu(np.stack([und, und[:, ::-1]], 1).reshape(-1, 2).T)
    rng = np.random.default_rng(8)
    pos_ids = np.sort(rng.choice(und.shape[0], 40, replace=False))
    neg = rng.integers(0, n, (30, 2))
    neg = neg[neg[:, 0] != neg[:, 1]]
    pairs = np.concatenate([und[pos_ids], neg])
    ptr, adj = ops.simple_adjacency(ei[0], ei[1], n)
    ei_new, x_new, _ = sample_block(double(cu(pos_ids), for_index=True), n, ei, None)
    mask = ops.adjacency_pair_mask(ptr, adj, cu(und[pos_ids, 0]), cu(und[pos_ids, 1]))
    cn = ops.common_neighbors(ptr, adj, cu(pairs[:, 0]), cu(pairs[:, 1]), mask)
    keep = np.ones(ei.shape[1], bool)
    keep[2 * pos_ids], keep[2 * pos_ids + 1] = False, False
    return dict(n=n, ei=ei.cpu().numpy(), keep=keep, pairs=pairs, deleted=und[pos_ids], hp=hp, ha=ha, ei_new=ei_new, x_new=x_new,
                cn=cn, max_x=int(np.diff(hp).max()))


def ref_ncn(mod, b, feat, detach=()):
    """float64 NCN on the CPU from mod's state_dict -> (logits, {name: leaf parameter}). detach: pair terms ("ij", "cn") whose
    gradient to the encoder is dropped - a reference that the gradient check must tell apart from the true one."""
    from oracle import twowl_oracle as O
    P = {k: v.detach().cpu().double().requires_grad_() for k, v in mod.state_dict().items()}
    ei = torch.from_numpy(b["ei"][:, b["keep"]])
    n = b["n"]
    if feat is None:
        deg = torch.bincount(ei[0], minlength=n).clamp(max=mod.max_x)
        h = P["emb.weight"][deg]
    else:
        h = feat.cpu().double()
    for i in range(len(mod.convs)):
        h = O.gcn_conv(h, ei, P[f"convs.{i}.lin.weight"], P[f"convs.{i}.bias"])
        if i < len(mod.convs) - 1:
            h = torch.relu(h)
    u, v = (torch.from_numpy(b["pairs"][:, k]) for k in (0, 1))
    lin = lambda name, x: x @ P[f"{name}.weight"].t() + P[f"{name}.bias"]   # noqa: E731
    hp = h.detach() if "ij" in detach else h
    r = torch.relu(lin("lin_ij", hp[u] * hp[v]))
    if mod.cn:
        dp, da = deleted_graph(b["hp"], b["ha"], b["deleted"])
        A = sp.csr_matrix((np.ones(da.size), da.astype(np.int64), dp), shape=(n, n))
        Cm = torch.from_numpy(A[b["pairs"][:, 0]].multiply(A[b["pairs"][:, 1]]).toarray())    # [B, n] common-neighbour indicator
        r = torch.cat((r, torch.relu(lin("lin_cn", Cm @ (h.detach() if "cn" in detach else h)))), 1)
    z = torch.relu(lin("lin_h", r))
    return lin("lin_o", z), P


# ||got - ref|| <= NCN_REL ||ref|| per tensor. The same restatement evaluated in float32 on the CPU stays within 1.2e-6 of float64
# on every tensor of this test; a halved gradient is off by 0.5, and dropping one pair term's gradient to the encoder by 0.17 or more.
NCN_REL = 1e-4


def _rel_err(got, ref) -> float:
    ref = torch.zeros(got.shape, dtype=torch.float64) if ref is None else ref.detach()
    return float((got.detach().cpu().double() - ref).norm() / ref.norm().clamp(min=1e-300))


@pytest.mark.gpu
@pytest.mark.parametrize("cn_term", [True, False])
@pytest.mark.parametrize("F", [0, 6])
def test_ncn_against_float64_restatement(ops, cn_term, F):
    from TwoWL.model.ncn import NCN
    b = _ncn_batch(ops)
    torch.manual_seed(0)
    mod = NCN(b["max_x"], hidden=16, num_layers=2, dropout=0.0, cn=cn_term, node_feat_dim=F).cuda().train()
    feat = torch.randn((b["n"], F)).cuda() if F else None
    w = torch.randn((b["pairs"].shape[0], 1))
    out = mod(b["x_new"], b["ei_new"], cu(b["pairs"]), b["cn"] if cn_term else None, feat)
    (out * w.cuda()).sum().backward()
    o64, P = ref_ncn(mod, b, feat)
    (o64 * w.double()).sum().backward()
    assert _rel_err(out, o64) <= NCN_REL, ("logits", _rel_err(out, o64))
    grads = {name: p.grad for name, p in mod.named_parameters()}
    assert set(grads) == set(P)
    for name, g in grads.items():
        assert _rel_err(g, P[name].grad) <= NCN_REL, (name, _rel_err(g, P[name].grad))
        # the check can fail: a halved or zeroed gradient is rejected
        assert _rel_err(0.5 * g, P[name].grad) > NCN_REL and _rel_err(0 * g, P[name].grad) > NCN_REL, name
    # ... and so is a reference whose pair terms send nothing back to the encoder: the encoder's gradients see both terms
    enc = [name for name in grads if name.startswith(("convs.", "emb."))]
    for term in ("ij",) + (("cn",) if cn_term else ()):
        o_d, P_d = ref_ncn(mod, b, feat, detach=(term,))
        (o_d * w.double()).sum().backward()
        assert any(_rel_err(grads[name], P_d[name].grad) > NCN_REL for name in enc), f"the {term} term's gradient is not seen"


@pytest.mark.gpu
def test_ncn_dropout_repeatable(ops):
    from TwoWL.model.ncn import NCN
    b = _ncn_batch(ops)
    torch.manual_seed(0)
    mod = NCN(b["max_x"], hidden=16, dropout=0.5).cuda().train()
    pairs = cu(b["pairs"])
    res = []
    for _ in range(2):
        mod.zero_grad()
        out = mod(b["x_new"], b["ei_new"], pairs, b["cn"], seed=12345)
        out.sum().backward()
        res.append([out.detach().clone()] + [p.grad.clone() for p in mod.parameters()])
    assert all(torch.equal(x, y) for x, y in zip(*res))
    mod.zero_grad()
    assert not torch.equal(mod(b["x_new"], b["ei_new"], pairs, b["cn"], seed=777).detach(), res[0][0])


# ------------------------------------------------------------------------------ training, scores, re-ranking

@pytest.mark.gpu
def test_ncn_fit_repeatable_and_scores_batch_independent(fbg):
    from TwoWL.model.train import ncn_fit, ncn_scores
    D, bg, _ = fbg
    trn, tst = D.dataset(*bg.split(0)), D.dataset(*bg.split(2))
    runs = [ncn_fit(trn, 1, 256, seed=4) for _ in range(2)]
    (m0, l0), (m1, l1) = runs
    assert torch.equal(l0, l1) and l0.numel() > 0 and bool(torch.isfinite(l0).all())
    for (k0, a), (k1, b) in zip(m0.state_dict().items(), m1.state_dict().items()):
        assert k0 == k1 and torch.equal(a, b), k0
    s = ncn_scores(m0, tst)
    assert s.shape == (tst.y.shape[0] // 2,) and s.dtype == torch.float32 and bool(torch.isfinite(s).all())
    assert torch.equal(s, ncn_scores(m0, tst, batch_size=37))
    g, _ = ncn_fit(trn, 1, 256, cn=False, seed=4)
    assert torch.equal(ncn_scores(g, tst), ncn_scores(g, tst, batch_size=37))


@pytest.mark.gpu
def test_rerank_scores_reproduce_rerank(fbg):
    from TwoWL.model.train import ncn_fit, ncn_scores, recommend, rerank, rerank_scores
    D, bg, mod = fbg
    tst = D.dataset(*bg.split(2))
    E, P = tst.ei.shape[1], tst.y.shape[0] // 2
    src = tst.pos1[E::2][:P][tst.y.reshape(-1)[0::2] > 0.5][:100, 0].contiguous()
    ids, _ = recommend(tst, src, k=20, by="aa")
    ds = D.candidate_dataset(bg, 2, src, ids)
    targets = E + torch.arange(ds.y.shape[0], device="cuda")
    with torch.no_grad():
        logits = mod(ds.x, ds.ei, ds.pos1, targets, ds.ei2, True)
    rid, rlog = rerank(mod, ds)
    sid, slog = rerank_scores(logits, ds)
    assert torch.equal(rid, sid) and torch.equal(rlog.view(torch.int32), slog.view(torch.int32))
    # NCN re-ranks the same shortlist: a permutation of each row, scores descending, padding last
    ncn, _ = ncn_fit(D.dataset(*bg.split(0)), 1, 256)
    nid, nlog = rerank_scores(ncn_scores(ncn, ds), ds)
    assert torch.equal(torch.sort(nid, 1).values, torch.sort(ids, 1).values)
    assert bool((nlog[:, :-1] >= nlog[:, 1:]).all()) and bool(((nid < 0) == torch.isinf(nlog)).all())


# measured on one B200 (1000 W power limit) with these settings: test AUC 0.901 (gcn 0.872, CN 0.845, SEAL 0.925); the floor sits
# 0.041 below it
NCN_FB = dict(epochs=40, batch_size=256, lr=5e-3, seed=0)
AUC_FLOOR = 0.86


@pytest.mark.gpu
def test_ncn_end_to_end_fb_pages_food(fbg):
    import time
    from TwoWL.model.train import heuristic_scores, ncn_fit, ncn_scores, rank_scores
    from twowl_b200 import ops
    D, bg, _ = fbg
    trn, tst = D.dataset(*bg.split(0)), D.dataset(*bg.split(2))
    labels = tst.y.reshape(-1)[0::2]
    table = {}
    for name, cn_term in (("ncn", True), ("gcn", False)):
        t0 = time.perf_counter()
        mod, losses = ncn_fit(trn, cn=cn_term, **NCN_FB)
        torch.cuda.synchronize()
        secs = time.perf_counter() - t0
        s = ncn_scores(mod, tst)
        assert losses[-1] < losses[0], name
        table[name] = (float(ops.auc(s, labels)[0]), rank_scores(s, tst, (20, 50, 100)))
        print(f"{name} training {secs:.2f} s, {losses.numel()} steps, loss {float(losses[0]):.4f} -> {float(losses[-1]):.4f}")
    table["cn"] = (float(ops.auc(heuristic_scores(tst)["cn"], labels)[0]), rank_scores(heuristic_scores(tst)["cn"], tst, (20, 50, 100)))
    for name, (auc, rk) in table.items():
        print(f"fb-pages-food test {name}: AUC {auc:.4f} " + " ".join(f"{k} {v:.4f}" for k, v in rk.items()))
    assert table["ncn"][0] > AUC_FLOOR, table["ncn"][0]
