"""Link recommendation: twowl_recommend_plan + twowl_recommend (ops.recommend_links), TwoWL.model.train.recommend / rerank and
TwoWL.operators.datasets.candidate_dataset.

The reference is a numpy restatement of the contract: per source s, expand (v, w) for w in N(s) ascending and v in N(w)
ascending, drop v = s and v in N(s), group by v, sum the aa / ra terms over each group in ascending w order one float64
addition at a time, and order the candidates by (-score, id). cn is an integer, jaccard the fp32 quotient of two integers and
ra a float64 sum of correctly rounded quotients in a fixed order: all three are EQUAL to the restatement, and so are the ids
ranked by them. aa's terms go through the device log, so aa lies within 0.5 ulp32 + 2 c 2^-53 of the float64 sum (the
heuristics tests' bound), and its ids are equal except where adjacent candidates' float64 scores lie within that bound."""
import numpy as np
import pytest
import torch

from test_gpu_heuristics import FAKE, EINVAL, ENOSPC, L, _err, cu, np_adjacency  # noqa: F401  (L is a fixture)

HEURISTICS = ("cn", "jaccard", "aa", "ra")


# ------------------------------------------------------------------------------ CPU: argument checks of the C ABI

def test_recommend_plan_argument_errors(L):
    lib = L.lib
    f = lib.twowl_recommend_plan
    nb = lib.twowl_recommend_plan_workspace_bytes(1000)
    assert nb >= lib.twowl_recommend_plan_workspace_bytes(0) > 0
    _err(L, f(FAKE, FAKE, 50, FAKE, 1, -1, FAKE, FAKE, FAKE, nb, None), EINVAL, "bad sizes")
    _err(L, f(FAKE, FAKE, 50, FAKE, 1, 1 << 31, FAKE, FAKE, FAKE, nb, None), EINVAL, "bad sizes")
    _err(L, f(FAKE, FAKE, -1, FAKE, 1, 1000, FAKE, FAKE, FAKE, nb, None), EINVAL, "bad sizes")
    _err(L, f(None, FAKE, 50, FAKE, 1, 1000, FAKE, FAKE, FAKE, nb, None), EINVAL, "null pointer")
    _err(L, f(FAKE, FAKE, 50, None, 1, 1000, FAKE, FAKE, FAKE, nb, None), EINVAL, "null pointer")
    _err(L, f(FAKE, FAKE, 50, FAKE, 1, 1000, None, FAKE, FAKE, nb, None), EINVAL, "null pointer")
    _err(L, f(FAKE, FAKE, 50, FAKE, 1, 1000, FAKE, None, FAKE, nb, None), EINVAL, "null pointer")
    _err(L, f(FAKE, FAKE, 50, FAKE, 1, 1000, FAKE, FAKE, FAKE, nb - 1, None), ENOSPC, "workspace too small")


def test_recommend_argument_errors(L):
    lib = L.lib
    f = lib.twowl_recommend
    nb = lib.twowl_recommend_workspace_bytes(5000, 100)
    assert nb > lib.twowl_recommend_workspace_bytes(0, 0) > 0
    assert lib.twowl_recommend_workspace_bytes(5000, 100) >= lib.twowl_recommend_workspace_bytes(4999, 100)

    def call(Q=100, q0=0, q1=100, m=5000, by=2, k=10, ptr=FAKE, adj=FAKE, src=FAKE, off=FAKE, ids=FAKE, sc=FAKE, ws=nb):
        return f(ptr, adj, 50, src, 1, Q, q0, q1, off, m, by, k, ids, sc, FAKE, ws, None)

    _err(L, call(q0=60, q1=40), EINVAL, "bad sizes")
    _err(L, call(q0=-1), EINVAL, "bad sizes")
    _err(L, call(q1=101), EINVAL, "bad sizes")
    _err(L, call(Q=-1, q1=0), EINVAL, "bad sizes")
    _err(L, call(k=0), EINVAL, "k must")
    _err(L, call(k=-3), EINVAL, "k must")
    _err(L, call(by=4), EINVAL, "by must")
    _err(L, call(by=-1), EINVAL, "by must")
    _err(L, call(m=-1), EINVAL, "n_entries")
    _err(L, call(m=1 << 31), EINVAL, "n_entries")
    for kw in ("ptr", "adj", "src", "off", "ids", "sc"):
        _err(L, call(**{kw: None}), EINVAL, "null pointer")
    _err(L, call(ws=nb - 1), ENOSPC, "workspace too small")


def test_recommend_links_refuses_cpu_tensors_and_bad_arguments(L):
    from twowl_b200 import ops
    ptr, adj, src = torch.zeros(6, dtype=torch.int64), torch.zeros(0, dtype=torch.int32), torch.zeros(3, dtype=torch.int64)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.recommend_links(ptr, adj, src, 5)
    for by in ("katz", "AA", ""):
        with pytest.raises(ValueError, match="by must"):
            ops.recommend_links(ptr, adj, src, 5, by=by)
    for k in (0, -1):
        with pytest.raises(ValueError, match="k must"):
            ops.recommend_links(ptr, adj, src, k)


# ------------------------------------------------------------------------------ numpy restatement

def _seq_sums(terms, start, cnt):
    """float64 sum of terms[start[i] : start[i] + cnt[i]] for every group i, added one at a time in order."""
    acc = np.zeros(cnt.size)
    order = np.argsort(-cnt, kind="stable")
    cs = cnt[order]
    for t in range(int(cs.max()) if cs.size else 0):
        act = order[:np.searchsorted(-cs, -t, side="left")]          # the groups with more than t terms
        acc[act] += terms[start[act] + t]
    return acc


def np_candidates(ptr, adj, s):
    """-> (v, c, jaccard fp32, aa float64, ra float64) of every candidate of s, v ascending."""
    d = np.diff(ptr)
    Ns = adj[ptr[s]:ptr[s + 1]].astype(np.int64)
    if Ns.size == 0:
        e = np.zeros(0)
        return np.zeros(0, np.int64), e, e.astype(np.float32), e, e
    lens = d[Ns]
    first = np.repeat(ptr[Ns] - np.concatenate(([0], np.cumsum(lens)[:-1])), lens)
    vs = adj[first + np.arange(lens.sum())].astype(np.int64)     # w ascending, then v ascending within N(w)
    ws = np.repeat(Ns, lens)
    keep = (vs != s) & ~np.isin(vs, Ns)
    vs, ws = vs[keep], ws[keep]
    o = np.argsort(vs, kind="stable")                             # stable: w stays ascending inside every v
    vs, ws = vs[o], ws[o]
    v, start, cnt = np.unique(vs, return_index=True, return_counts=True)
    dw = d[ws].astype(np.float64)
    with np.errstate(divide="ignore"):
        aa = _seq_sums(np.where(dw > 1, 1.0 / np.log(np.maximum(dw, 2)), 0.0), start, cnt)
    ra = _seq_sums(1.0 / dw, start, cnt)
    den = d[s] + d[v] - cnt
    jac = (np.float32(cnt) / den.astype(np.float32)).astype(np.float32)
    return v, cnt.astype(np.float64), jac, aa, ra


def np_recommend(ptr, adj, src, k, by):
    """-> (ids [Q, k], scores float64 [4, Q, k] with NaN padding, the full candidate tables per source)."""
    Q = len(src)
    ids = np.full((Q, k), -1, np.int64)
    sc = np.full((4, Q, k), np.nan)
    tables = []
    for q, s in enumerate(src):
        v, c, jac, aa, ra = np_candidates(ptr, adj, int(s))
        cols = (c, jac.astype(np.float64), aa, ra)
        key = cols[HEURISTICS.index(by)].astype(np.float32)     # the op orders by the fp32 score, as it returns it
        o = np.lexsort((v, -key))[:k]
        ids[q, :o.size] = v[o]
        for h in range(4):
            sc[h, q, :o.size] = cols[h][o]
        tables.append(dict(zip(v.tolist(), zip(*[x.tolist() for x in cols]))))
    return ids, sc, tables


def aa_tol(ref, c):
    return 0.5 * np.spacing(np.abs(ref).astype(np.float32)).astype(np.float64) + 2 * c * 2.0 ** -53 * np.abs(ref)


def check_recommend(ids, scores, ptr, adj, src, k, by, what):
    """ids / scores: the op's outputs (torch); the restatement's ids and bits as the module docstring states."""
    gi, gs = ids.cpu().numpy(), scores.cpu().numpy()
    ri, rs, tables = np_recommend(ptr, adj, src, k, by)
    assert gi.shape == (len(src), k) and gs.shape == (4, len(src), k), what
    valid = ri >= 0
    assert np.array_equal(gi >= 0, valid), f"{what}: candidate counts differ"
    assert np.isnan(gs[:, ~valid]).all(), f"{what}: padding is not NaN"
    if by != "aa":
        assert np.array_equal(gi, ri), f"{what}: ids differ at {np.argwhere(gi != ri)[:5].tolist()}"
    else:                   # equal except at near-ties: the float64 scores of the swapped candidates lie within the bound
        for q, j in np.argwhere(gi != ri):
            a, b = tables[q][int(gi[q, j])][2], tables[q][int(ri[q, j])][2]
            c = max(tables[q][int(gi[q, j])][0], tables[q][int(ri[q, j])][0])
            assert abs(a - b) <= 2 * aa_tol(np.array([max(a, b)]), c)[0], f"{what}: aa ids differ at ({q}, {j}) beyond a near-tie"
    # the scores of the returned ids, looked up in the restatement's tables
    want = np.full((4, len(src), k), np.nan)
    for q, j in np.argwhere(gi >= 0):
        want[:, q, j] = tables[q][int(gi[q, j])]
    for h, name in ((0, "cn"), (1, "jaccard"), (3, "ra")):
        assert np.array_equal(gs[h][valid], want[h][valid].astype(np.float32)), f"{what}: {name} bits differ"
    err, tol = np.abs(gs[2][valid].astype(np.float64) - want[2][valid]), aa_tol(want[2][valid], want[0][valid])
    assert (err <= tol).all(), f"{what}: aa off by {err[err > tol][:5]} > {tol[err > tol][:5]}"
    # each row is ordered by the chosen fp32 score descending, ties by id ascending
    h = HEURISTICS.index(by)
    for q in range(len(src)):
        m = int(valid[q].sum())
        key = gs[h, q, :m]
        assert (np.diff(key) <= 0).all() and all(gi[q, j] < gi[q, j + 1] for j in range(m - 1) if key[j] == key[j + 1]), \
            f"{what}: row {q} is out of order"
    return gi, gs


# ------------------------------------------------------------------------------ GPU

@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from twowl_b200 import ops as o
    return o


def _graph(ops, r, c, n):
    ptr, adj = ops.simple_adjacency(cu(r), cu(c), n)
    return ptr, adj, ptr.cpu().numpy(), adj.cpu().numpy()


def _check_graph(ops, r, c, n, Q, k, seed, what):
    """Q random sources plus the max-degree node (three times), an isolated node and up to 20 neighbours of the hub."""
    rng = np.random.default_rng(seed)
    ptr, adj, hp, ha = _graph(ops, r, c, n)
    deg = np.diff(hp)
    hub = int(np.argmax(deg))
    src = rng.integers(0, n, Q)
    src[:3] = hub
    iso = np.nonzero(deg == 0)[0]
    if iso.size:
        src[3] = iso[0]
    hub_nbrs = ha[hp[hub]:hp[hub + 1]]
    src[4:4 + min(20, hub_nbrs.size)] = hub_nbrs[:20]                  # sources adjacent to the hub
    tsrc = cu(src)
    outs = {}
    for by in HEURISTICS:
        ids, sc = ops.recommend_links(ptr, adj, tsrc, k, by=by)
        check_recommend(ids, sc, hp, ha, src, k, by, f"{what} by {by}")
        i2, s2 = ops.recommend_links(ptr, adj, tsrc, k, by=by)
        assert torch.equal(ids, i2) and torch.equal(sc.view(torch.int32), s2.view(torch.int32)), f"{what} by {by}: not repeatable"
        outs[by] = (ids, sc)
    # every returned pair scores the same under link_heuristics (cn / jaccard bits; aa / ra within the bound: another order)
    ids, sc = outs["aa"]
    m = ids >= 0
    u = tsrc.unsqueeze(1).expand_as(ids)[m]
    lh = ops.link_heuristics(ptr, adj, u, ids[m]).cpu().numpy()
    got = sc[:, m].cpu().numpy()
    assert np.array_equal(lh[0], got[0]) and np.array_equal(lh[1], got[1]), f"{what}: cn / jaccard differ from link_heuristics"
    for h in (2, 3):
        ref = lh[h].astype(np.float64)
        assert (np.abs(got[h] - ref) <= 2 * aa_tol(ref, lh[0]) + np.spacing(lh[h])).all(), f"{what}: row {h} far from link_heuristics"
    return ptr, adj, hp, ha, src, outs


@pytest.mark.gpu
def test_recommend_erdos_renyi(ops):
    rng = np.random.default_rng(11)
    n, m = 3000, 18000
    r, c = rng.integers(0, n - 100, m), rng.integers(0, n - 100, m)     # the last 100 nodes are isolated
    _check_graph(ops, r, c, n, 300, 50, 12, "Erdos-Renyi")


@pytest.mark.gpu
def test_recommend_rmat_with_hubs(ops):
    from TwoWL.operators.synthetic import rmat_edges
    s, d, n = rmat_edges(12, 40_000, (0.57, 0.19, 0.19, 0.05), 13, torch.device("cuda"))
    ptr, adj, hp, ha, src, outs = _check_graph(ops, s.cpu().numpy(), d.cpu().numpy(), n, 300, 100, 14, "R-MAT")
    deg = np.diff(hp)
    assert deg.max() > 300
    # batching: one source per batch, and a budget below a single source's expansion, give the same bits as the default
    tsrc = cu(src)
    X = np.array([deg[ha[hp[x]:hp[x + 1]]].sum() for x in src])
    for budget in (1, int(X.max()) // 3, int(X.sum()) // 7):
        for by in ("cn", "aa"):
            ids, sc = ops.recommend_links(ptr, adj, tsrc, 100, by=by, max_entries=budget)
            assert torch.equal(ids, outs[by][0]) and torch.equal(sc.view(torch.int32), outs[by][1].view(torch.int32)), (budget, by)


@pytest.mark.gpu
def test_recommend_edge_cases(ops):
    rng = np.random.default_rng(15)
    n = 400
    # a hub (node 0) joined to 300 nodes, a sparse background among nodes 1..349, nodes 350..399 isolated except a path
    r = np.concatenate((np.zeros(300, np.int64), rng.integers(1, 350, 600), [360, 361]))
    c = np.concatenate((np.arange(1, 301), rng.integers(1, 350, 600), [361, 362]))
    ptr, adj, hp, ha = _graph(ops, r, c, n)
    few = 360                                                           # the path 360 - 361 - 362: one candidate
    src = np.array([0, 1, 2, few, 399, 0, 5, 5, 399])                   # hub, hub neighbours, few, isolated, duplicates
    for k in (1, 7, n + 10):                                            # k > N
        for by in HEURISTICS:
            ids, sc = ops.recommend_links(ptr, adj, cu(src), k, by=by)
            gi, gs = check_recommend(ids, sc, hp, ha, src, k, by, f"edge cases k={k} by {by}")
            assert (gi[4] == -1).all() and np.isnan(gs[:, 4]).all()    # isolated
            assert gi[3, 0] == 362 and (gi[3, 1:] == -1).all()        # fewer than k candidates: padded
            assert np.array_equal(gi[0], gi[5]) and np.array_equal(gi[6], gi[7])
            assert np.array_equal(gs[:, 6].view(np.int32), gs[:, 7].view(np.int32))
    ids, sc = ops.recommend_links(ptr, adj, cu(src)[:0], 5)
    assert ids.shape == (0, 5) and sc.shape == (4, 0, 5)
    for bad in (-1, n, 1 << 40):
        b = src.copy()
        b[2] = bad
        with pytest.raises(IndexError, match="outside"):
            ops.recommend_links(ptr, adj, cu(b), 5)
    # a strided source view
    two = cu(np.stack((src, src), axis=1))
    i1, s1 = ops.recommend_links(ptr, adj, two[:, 1], 7)
    i2, s2 = ops.recommend_links(ptr, adj, cu(src), 7)
    assert torch.equal(i1, i2) and torch.equal(s1.view(torch.int32), s2.view(torch.int32))
    # an empty graph: every row is padding
    p0, a0 = ops.simple_adjacency(cu(np.zeros(0)), cu(np.zeros(0)), 7)
    i0, s0 = ops.recommend_links(p0, a0, cu([0, 3, 6]), 4)
    assert (i0 == -1).all() and s0.isnan().all()
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------ GPU: end to end on fb-pages-food

@pytest.fixture(scope="module")
def fbg(fb):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import TwoWL.model.model as model
    import TwoWL.operators.datasets as D
    from helpers import state_dict_from
    from test_gpu_ranking import CFG1
    n = int(fb["num_nodes"][0])
    ep, en = (torch.from_numpy(fb[k].astype(np.int64)).cuda() for k in ("edge_pos", "edge_neg"))
    bg = D.BaseGraph(torch.zeros((n, 0), device="cuda"), None, ep, en, torch.from_numpy(fb["num_pos"]),
                     torch.from_numpy(fb["num_neg"]), "2wl_l")
    bg.preprocess()
    bg.setPosDegreeFeature()
    sd = state_dict_from(fb)
    mod = model.LocalWLNet(sd["emb.0.weight"].shape[0] - 1, False, None, **CFG1)
    mod.load_state_dict(sd, strict=True)
    return D, bg, mod.cuda().eval()


@pytest.mark.gpu
def test_recommend_and_rerank_fb_pages_food(fbg):
    from TwoWL.model.train import recommend, rerank
    from TwoWL.utils import get_ei2
    D, bg, mod = fbg
    n = bg.num_nodes
    tst = D.dataset(*bg.split(2))
    E = tst.ei.shape[1]
    P = tst.y.shape[0] // 2
    pos = tst.pos1[E::2][:P][tst.y.reshape(-1)[0::2] > 0.5]
    src = pos[:200, 0].contiguous()
    ei = tst.ei.cpu().numpy()
    hp, ha = np_adjacency(ei[0], ei[1], n)
    for by in HEURISTICS:
        ids, sc = recommend(tst, src, k=20, by=by)
        check_recommend(ids, sc, hp, ha, src.cpu().numpy(), 20, by, f"fb-pages-food by {by}")
    ids, sc = recommend(tst, src, k=20, by="aa")
    ds = D.candidate_dataset(bg, 2, src, ids)
    # the table, hand-built for the same pairs
    m = ids >= 0
    pairs = torch.stack((src.unsqueeze(1).expand_as(ids)[m], ids[m]))
    pred = torch.stack((pairs, pairs.flip(0)), dim=2).reshape(2, -1)
    assert torch.equal(ds.pos1, torch.cat((tst.ei.t(), pred.t()), dim=0))
    assert torch.equal(ds.ei2, get_ei2(n, tst.ei, pred))
    assert torch.equal(ds.x, tst.x) and torch.equal(ds.ei, tst.ei) and ds.y.shape == (pred.shape[1], 1) and not ds.y.any()
    assert torch.equal(ds.cand_mask, m) and torch.equal(ds.cand_ids, ids)
    # rerank: the model's logits on that table, each row ordered by logit descending, ties in the heuristic's order, padding last
    rid, rlog = rerank(mod, ds)
    targets = E + torch.arange(ds.y.shape[0], device="cuda")
    with torch.no_grad():
        logits = mod(ds.x, ds.ei, ds.pos1, targets, ds.ei2, True).reshape(-1)
    table = np.full(ids.shape, -np.inf, np.float32)
    table[m.cpu().numpy()] = logits.cpu().numpy()
    hid = ids.cpu().numpy()
    for q in range(ids.shape[0]):
        o = np.lexsort((np.arange(ids.shape[1]), -table[q]))
        assert np.array_equal(rid[q].cpu().numpy(), hid[q, o]), q
        assert np.array_equal(rlog[q].cpu().numpy().view(np.int32), table[q, o].view(np.int32)), q
    with pytest.raises(ValueError, match="split"):
        D.candidate_dataset(bg, 3, src, ids)
