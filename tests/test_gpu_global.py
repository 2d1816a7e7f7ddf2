"""Global link-prediction heuristics: twowl_walk_scale / restart / gather / topk around seg_reduce (ops.global_heuristics,
ops.recommend_global), TwoWL.model.train.global_heuristic_scores / recommend_global.

The reference is a scipy float64 restatement of the recursions with the fp32-rounded damping:
  Katz: y_0 = 0, y_{t+1} = A (beta (y_t + e_s));  PPR: pi_0 = e_s, pi_{t+1} = A ((alpha / d) pi_t) + (1 - alpha) e_s.
Every term is >= 0, so one step's relative error at row v is at most gamma_{d(v)+2} (the sum, the scale quotient, the restart
add), gamma_n = n u / (1 - n u), u = 2^-24; over L steps (1 + gamma_{dmax+2})^L - 1. Where the float64 score is 0 (v not reached)
the device gives exactly 0. PPR paths through hubs fall below fp32's normal range, so the bound has an absolute floor of
4 x 2^-126: a score that underflows to 0 is not a candidate."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

from test_gpu_heuristics import FAKE, EINVAL, ENOSPC, L, _err, cu, np_adjacency  # noqa: F401  (L is a fixture)
from test_gpu_recommend import fbg  # noqa: F401  (a fixture: fb-pages-food's graph and the reference model)

FLOOR = 4 * 2.0 ** -126
DEFAULTS = {"katz": (3, 0.001), "ppr": (20, 0.85)}


# ------------------------------------------------------------------------------ CPU: argument checks of the C ABI

def test_walk_scale_restart_gather_argument_errors(L):
    lib = L.lib
    f = lib.twowl_walk_scale
    _err(L, f(FAKE, -1, 0, 0.5, FAKE, None), EINVAL, "bad sizes")
    _err(L, f(FAKE, 1 << 31, 0, 0.5, FAKE, None), EINVAL, "bad sizes")
    for m in (-1, 2):
        _err(L, f(FAKE, 10, m, 0.5, FAKE, None), EINVAL, "method must")
    for m, d in ((0, 0.0), (0, -1.0), (0, float("inf")), (0, float("nan")), (1, 0.0), (1, 1.0), (1, 1.5), (1, float("nan"))):
        _err(L, f(FAKE, 10, m, d, FAKE, None), EINVAL, "damping must")
    _err(L, f(None, 10, 0, 0.5, FAKE, None), EINVAL, "null pointer")
    _err(L, f(FAKE, 10, 1, 0.5, None, None), EINVAL, "null pointer")

    f = lib.twowl_walk_restart
    _err(L, f(FAKE, 68, 10, FAKE, 1, -1, 1.0, None), EINVAL, "bad sizes")
    _err(L, f(FAKE, 8, 10, FAKE, 1, 9, 1.0, None), EINVAL, "bad sizes")
    _err(L, f(FAKE, 68, -1, FAKE, 1, 4, 1.0, None), EINVAL, "bad sizes")
    _err(L, f(None, 68, 10, FAKE, 1, 4, 1.0, None), EINVAL, "null pointer")
    _err(L, f(FAKE, 68, 10, None, 1, 4, 1.0, None), EINVAL, "null pointer")

    f = lib.twowl_walk_gather

    def gather(ld=68, n=10, P=5, c0=0, c1=4, Y=FAKE, col=FAKE, v=FAKE, dst=FAKE, out=FAKE):
        return f(Y, ld, n, col, v, dst, P, c0, c1, out, None)

    _err(L, gather(P=-1), EINVAL, "bad sizes")
    _err(L, gather(c0=-1), EINVAL, "bad sizes")
    _err(L, gather(c0=5, c1=4), EINVAL, "bad sizes")
    _err(L, gather(c1=69), EINVAL, "bad sizes")
    _err(L, gather(n=-1), EINVAL, "bad sizes")
    for kw in ("Y", "col", "v", "dst", "out"):
        _err(L, gather(**{kw: None}), EINVAL, "null pointer")


def test_walk_topk_argument_errors(L):
    lib = L.lib
    f = lib.twowl_walk_topk
    nb = lib.twowl_walk_topk_workspace_bytes(1000, 64, 100)
    assert nb > lib.twowl_walk_topk_workspace_bytes(1000, 64, 10) > 0
    assert lib.twowl_walk_topk_workspace_bytes(1000, 64, 2000) == lib.twowl_walk_topk_workspace_bytes(1000, 64, 1000)   # k > N

    def call(n=1000, ld=68, nc=64, k=100, Q=200, q0=0, ptr=FAKE, adj=FAKE, Y=FAKE, src=FAKE, ids=FAKE, sc=FAKE, ws=nb):
        return f(ptr, adj, n, Y, ld, src, 1, nc, k, Q, q0, ids, sc, FAKE, ws, None)

    _err(L, call(nc=-1), EINVAL, "bad sizes")
    _err(L, call(nc=69), EINVAL, "bad sizes")
    _err(L, call(n=-1), EINVAL, "bad sizes")
    _err(L, call(q0=-1), EINVAL, "bad sizes")
    _err(L, call(q0=137), EINVAL, "bad sizes")
    _err(L, call(k=0), EINVAL, "k must")
    _err(L, call(k=-2), EINVAL, "k must")
    _err(L, call(n=1 << 30, nc=64, k=1 << 26, ws=1 << 62), EINVAL, "n_cols * min")
    for kw in ("ptr", "Y", "src", "ids", "sc"):
        _err(L, call(**{kw: None}), EINVAL, "null pointer")
    _err(L, call(ws=nb - 1), ENOSPC, "workspace too small")


def test_global_ops_refuse_cpu_tensors_and_bad_arguments(L):
    from twowl_b200 import ops
    ptr, adj, u = torch.zeros(6, dtype=torch.int64), torch.zeros(0, dtype=torch.int32), torch.zeros(3, dtype=torch.int64)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.global_heuristics(ptr, adj, u, u)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.recommend_global(ptr, adj, u, 5)
    calls = (lambda **kw: ops.global_heuristics(ptr, adj, u, u, **kw), lambda **kw: ops.recommend_global(ptr, adj, u, 5, **kw))
    for fn in calls:
        for by in ("aa", "KATZ", "", "pagerank"):
            with pytest.raises(ValueError, match="by must"):
                fn(by=by)
        for by in ("katz", "ppr"):
            for steps in (0, -1):
                with pytest.raises(ValueError, match="steps must"):
                    fn(by=by, steps=steps)
        for beta in (0.0, -0.1, float("inf"), float("nan"), 1e300):
            with pytest.raises(ValueError, match="beta"):
                fn(by="katz", damping=beta)
        for alpha in (0.0, 1.0, -0.5, 1.5, float("nan")):
            with pytest.raises(ValueError, match="alpha"):
                fn(by="ppr", damping=alpha)
        for mc in (0, 1025):
            with pytest.raises(ValueError, match="max_cols"):
                fn(max_cols=mc)
    for k in (0, -1):
        with pytest.raises(ValueError, match="k must"):
            ops.recommend_global(ptr, adj, u, k)


# ------------------------------------------------------------------------------ float64 restatement

def np_walk(ptr, adj, src, by, steps, damping):
    """float64 scores [len(src), N] of every node from each source, the damping rounded to fp32 first."""
    n = len(ptr) - 1
    A = sp.csr_matrix((np.ones(len(adj)), adj.astype(np.int64), ptr), shape=(n, n))
    d = np.diff(ptr).astype(np.float64)
    E = np.zeros((n, len(src)))
    E[np.asarray(src, np.int64), np.arange(len(src))] = 1.0
    p = float(np.float32(damping))
    if by == "katz":
        Y = np.zeros((n, len(src)))
        for _ in range(steps):
            Y = A @ (p * (Y + E))
    else:
        sc = np.where(d > 0, p / np.maximum(d, 1), 0.0)[:, None]
        r = float(np.float32(1) - np.float32(p))
        Y = E.copy()
        for _ in range(steps):
            Y = A @ (sc * Y) + r * E
    return Y.T


def bound(ptr, steps):
    u = 2.0 ** -24
    m = int(np.diff(ptr).max(initial=0)) + 2
    return (1 + m * u / (1 - m * u)) ** steps - 1


def check_bound(got, ref, ptr, steps, what):
    got = np.asarray(got, np.float64)
    assert np.array_equal(got[ref == 0], np.zeros(int((ref == 0).sum()))), f"{what}: a node not reached scores != 0"
    err, tol = np.abs(got - ref), bound(ptr, steps) * ref + FLOOR
    assert (err <= tol).all(), f"{what}: off by {err[err > tol][:5]} > {tol[err > tol][:5]}"


def np_topk(full, ptr, adj, src, k):
    """The contract's top-k of the device's own scores [Q, N]: s and N(s) removed, score > 0, order (-score, id)."""
    Q, n = full.shape
    ids = np.full((Q, k), -1, np.int64)
    sc = np.full((Q, k), np.nan, np.float32)
    for q, s in enumerate(src):
        keep = full[q] > 0
        keep[s] = False
        keep[adj[ptr[s]:ptr[s + 1]]] = False
        v = np.nonzero(keep)[0]
        o = v[np.lexsort((v, -full[q, v]))][:k]
        ids[q, :o.size] = o
        sc[q, :o.size] = full[q, o]
    return ids, sc


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


def _sources(rng, hp, ha, Q):
    """Q random nodes, the max-degree node, an isolated node (if any), up to 10 neighbours of the hub, one duplicate."""
    deg = np.diff(hp)
    hub = int(np.argmax(deg))
    src = rng.integers(0, len(deg), Q)
    src[0] = src[1] = hub
    iso = np.nonzero(deg == 0)[0]
    if iso.size:
        src[2] = iso[0]
    nb = ha[hp[hub]:hp[hub + 1]][:10]
    src[3:3 + nb.size] = nb
    return src


def _full(ops, ptr, adj, src, n, **kw):
    """global_heuristics(s, v) for every v, rows in src order -> fp32 [Q, N] (numpy)."""
    u = cu(np.repeat(src, n))
    v = cu(np.tile(np.arange(n), len(src)))
    return ops.global_heuristics(ptr, adj, u, v, **kw).cpu().numpy().reshape(len(src), n)


def _check_graph(ops, r, c, n, seed, what, Q=24, k=60):
    rng = np.random.default_rng(seed)
    ptr, adj, hp, ha = _graph(ops, r, c, n)
    src = _sources(rng, hp, ha, Q)
    for by, steps_list, damps in (("katz", (1, 2, 3, 5), (None, 0.05)), ("ppr", (1, 5, 20), (None, 0.5))):
        for steps in steps_list:
            for damp in damps:
                tag = f"{what} {by} L={steps} damping={damp}"
                full = _full(ops, ptr, adj, src, n, by=by, steps=steps, damping=damp)
                ref = np_walk(hp, ha, src, by, steps, DEFAULTS[by][1] if damp is None else damp)
                check_bound(full, ref, hp, steps, tag)
                ids, sc = ops.recommend_global(ptr, adj, cu(src), k, by=by, steps=steps, damping=damp)
                gi, gs = ids.cpu().numpy(), sc.cpu().numpy()
                ri, rs = np_topk(full, hp, ha, src, k)
                assert np.array_equal(gi, ri), f"{tag}: ids differ at {np.argwhere(gi != ri)[:5].tolist()}"
                valid = gi >= 0
                assert np.array_equal(gs[valid].view(np.int32), rs[valid].view(np.int32)), f"{tag}: score bits differ"
                assert np.isnan(gs[~valid]).all(), f"{tag}: padding is not NaN"
                # against float64: where the ids differ from its order, the two candidates' float64 scores are a near-tie
                fi, _ = np_topk(ref, hp, ha, src, k)
                tol = bound(hp, steps)
                for q, j in np.argwhere((gi != fi) & (gi >= 0) & (fi >= 0)):
                    a, b = ref[q, gi[q, j]], ref[q, fi[q, j]]
                    assert abs(a - b) <= 2 * (tol * max(a, b) + FLOOR), f"{tag}: ids differ at ({q}, {j}) beyond a near-tie"
    return ptr, adj, hp, ha, src


@pytest.mark.gpu
def test_global_erdos_renyi(ops):
    rng = np.random.default_rng(21)
    n, m = 2000, 8000
    r, c = rng.integers(0, n - 50, m), rng.integers(0, n - 50, m)       # the last 50 nodes are isolated
    _check_graph(ops, r, c, n, 22, "Erdos-Renyi")


def _rmat_with_hub(seed):
    """R-MAT on 4096 nodes (hubs near degree 1000) plus one node joined to 3000 others: a row of more than 32 chunks of 64,
    which seg_reduce combines with a whole CTA - the path whose lane-group count depends on the operand width below 68."""
    from TwoWL.operators.synthetic import rmat_edges
    s, d, n = rmat_edges(12, 40_000, (0.57, 0.19, 0.19, 0.05), seed, torch.device("cuda"))
    rng = np.random.default_rng(seed)
    hub = int(rng.integers(0, n))
    others = rng.choice(np.setdiff1d(np.arange(n), [hub]), 3000, replace=False)
    r = np.concatenate((s.cpu().numpy(), np.full(others.size, hub)))
    c = np.concatenate((d.cpu().numpy(), others))
    return r, c, n


def _assert_long_rows(hp):
    deg = np.diff(hp)
    assert deg.max() > 32 * 64, "the hub must take seg_reduce's whole-CTA long-row path"
    assert ((deg > 64) & (deg <= 32 * 64)).sum() > 10, "rows on the one-group long-row path"


@pytest.mark.gpu
def test_global_rmat_with_hubs(ops):
    r, c, n = _rmat_with_hub(23)
    ptr, adj, hp, ha, src = _check_graph(ops, r, c, n, 24, "R-MAT")
    _assert_long_rows(hp)


@pytest.mark.gpu
def test_global_batching_and_repeatability(ops):
    r, c, n = _rmat_with_hub(25)
    ptr, adj, hp, ha = _graph(ops, r, c, n)
    _assert_long_rows(hp)
    rng = np.random.default_rng(26)
    src = _sources(rng, hp, ha, 300)
    v = rng.integers(0, n, src.size)
    for by in ("katz", "ppr"):
        base = ops.global_heuristics(ptr, adj, cu(src), cu(v), by=by)
        ids, sc = ops.recommend_global(ptr, adj, cu(src), 50, by=by)
        again = ops.global_heuristics(ptr, adj, cu(src), cu(v), by=by)
        i2, s2 = ops.recommend_global(ptr, adj, cu(src), 50, by=by)
        assert torch.equal(base.view(torch.int32), again.view(torch.int32)) and torch.equal(ids, i2) and \
            torch.equal(sc.view(torch.int32), s2.view(torch.int32)), f"{by}: not repeatable"
        for mc in (4, 17, 300, 1024):
            g = ops.global_heuristics(ptr, adj, cu(src), cu(v), by=by, max_cols=mc)
            assert torch.equal(g.view(torch.int32), base.view(torch.int32)), (by, mc)
            i3, s3 = ops.recommend_global(ptr, adj, cu(src), 50, by=by, max_cols=mc)
            assert torch.equal(i3, ids) and torch.equal(s3.view(torch.int32), sc.view(torch.int32)), (by, mc)
        # shuffled and duplicated sources: the same rows
        perm = rng.permutation(src.size)
        dup = np.concatenate((perm, perm[:40]))
        i4, s4 = ops.recommend_global(ptr, adj, cu(src[dup]), 50, by=by)
        assert torch.equal(i4, ids[cu(dup)]) and torch.equal(s4.view(torch.int32), sc[cu(dup)].view(torch.int32)), by
        g = ops.global_heuristics(ptr, adj, cu(src[dup]), cu(v[dup]), by=by, max_cols=8)
        assert torch.equal(g.view(torch.int32), base[cu(dup)].view(torch.int32)), by
        # recommend_global's scores are global_heuristics' bits for the same pairs
        m = ids >= 0
        uu = cu(src).unsqueeze(1).expand_as(ids)[m]
        assert torch.equal(ops.global_heuristics(ptr, adj, uu, ids[m], by=by).view(torch.int32), sc[m].view(torch.int32)), by
    # a ranking_dataset-shaped input: one source repeated 1 + k times, against one call per pair
    hub = int(np.argmax(np.diff(hp)))
    for s0 in (hub, int(src[5])):
        partners = rng.integers(0, n, 21)
        for by in ("katz", "ppr"):
            g = ops.global_heuristics(ptr, adj, cu(np.full(21, s0)), cu(partners), by=by).cpu().numpy()
            one = np.array([ops.global_heuristics(ptr, adj, cu([s0]), cu([p]), by=by).item() for p in partners], np.float32)
            assert np.array_equal(g.view(np.int32), one.view(np.int32)), (s0, by)


@pytest.mark.gpu
def test_global_edge_cases(ops):
    rng = np.random.default_rng(27)
    n = 400
    # a hub (node 0) joined to 300 nodes, a sparse background among 1..349, a path 360 - 361 - 362, nodes 363.. isolated
    r = np.concatenate((np.zeros(300, np.int64), rng.integers(1, 350, 600), [360, 361]))
    c = np.concatenate((np.arange(1, 301), rng.integers(1, 350, 600), [361, 362]))
    ptr, adj, hp, ha = _graph(ops, r, c, n)
    src = np.array([0, 1, 2, 360, 399, 0, 5, 5, 399])
    alpha = float(np.float32(0.85))
    for by in ("katz", "ppr"):
        for k in (1, 7, n + 10):                                            # k > N
            ids, sc = ops.recommend_global(ptr, adj, cu(src), k, by=by)
            gi, gs = ids.cpu().numpy(), sc.cpu().numpy()
            full = _full(ops, ptr, adj, src, n, by=by)
            ri, rs = np_topk(full, hp, ha, src, k)
            assert np.array_equal(gi, ri) and np.array_equal(gs[gi >= 0].view(np.int32), rs[gi >= 0].view(np.int32)), (by, k)
            assert np.isnan(gs[gi < 0]).all(), (by, k)
            assert (gi[4] == -1).all() and np.isnan(gs[4]).all()                        # isolated source: all padding
            assert gi[3, 0] == 362 and (gi[3, 1:] == -1).all()                          # the path: one candidate
            assert np.array_equal(gi[0], gi[5]) and np.array_equal(gs[6].view(np.int32), gs[7].view(np.int32))
        # u == v pairs; an isolated source's PPR mass stays at home: exactly 1 - alpha
        g = ops.global_heuristics(ptr, adj, cu([399, 0, 361]), cu([399, 0, 361]), by=by).cpu().numpy()
        ref = np_walk(hp, ha, [399, 0, 361], by, *DEFAULTS[by])
        check_bound(g, ref[np.arange(3), [399, 0, 361]], hp, DEFAULTS[by][0], f"{by} u == v")
        if by == "ppr":
            assert g[0] == np.float32(1) - np.float32(alpha)
        else:
            assert g[0] == 0
        # Q = 0 and P = 0
        i0, s0 = ops.recommend_global(ptr, adj, cu(src)[:0], 5, by=by)
        assert i0.shape == (0, 5) and s0.shape == (0, 5)
        assert ops.global_heuristics(ptr, adj, cu(src)[:0], cu(src)[:0], by=by).shape == (0,)
        # bad ids
        for bad in (-1, n, 1 << 40):
            b = src.copy()
            b[2] = bad
            with pytest.raises(IndexError, match="outside"):
                ops.recommend_global(ptr, adj, cu(b), 5, by=by)
            with pytest.raises(IndexError, match="outside"):
                ops.global_heuristics(ptr, adj, cu(b), cu(src), by=by)
            with pytest.raises(IndexError, match="outside"):
                ops.global_heuristics(ptr, adj, cu(src), cu(b), by=by)
        # a strided source view
        two = cu(np.stack((src, src), axis=1))
        i1, s1 = ops.recommend_global(ptr, adj, two[:, 1], 7, by=by)
        i2, s2 = ops.recommend_global(ptr, adj, cu(src), 7, by=by)
        assert torch.equal(i1, i2) and torch.equal(s1.view(torch.int32), s2.view(torch.int32))
        # an empty graph: Katz 0 everywhere, PPR 1 - alpha at (u, u); no candidates
        p0, a0 = ops.simple_adjacency(cu(np.zeros(0)), cu(np.zeros(0)), 7)
        g = ops.global_heuristics(p0, a0, cu([0, 3, 6, 2]), cu([0, 3, 5, 1]), by=by).cpu().numpy()
        want = np.array([1, 1, 0, 0], np.float32) * (np.float32(1) - np.float32(alpha)) if by == "ppr" else np.zeros(4, np.float32)
        assert np.array_equal(g, want), (by, g)
        i0, s0 = ops.recommend_global(p0, a0, cu([0, 3, 6]), 4, by=by)
        assert (i0 == -1).all() and s0.isnan().all()
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------ GPU: end to end on fb-pages-food

@pytest.mark.gpu
def test_global_end_to_end_fb_pages_food(fbg):
    from test_gpu_ranking import np_hits, np_rank
    from TwoWL.model.train import global_heuristic_scores, rank_scores, recommend, recommend_global, rerank
    from twowl_b200 import ops
    D, bg, mod = fbg
    n = bg.num_nodes
    tst = D.dataset(*bg.split(2))
    rk = D.ranking_dataset(bg, 2, num_neg=50)
    ks = (1, 10, 20, 50, 100)
    for ds, what in ((tst, "test split"), (rk, "ranking table")):
        E = ds.ei.shape[1]
        P = ds.y.shape[0] // 2
        ei = ds.ei.cpu().numpy()
        hp, ha = np_adjacency(ei[0], ei[1], n)
        pairs = ds.pos1[E::2][:P].cpu().numpy()
        for by in ("katz", "ppr"):
            s = global_heuristic_scores(ds, by)
            assert s.shape == (P,) and s.dtype == torch.float32
            if ds is tst:               # against float64: every distinct source's walk
                us, inv = np.unique(pairs[:, 0], return_inverse=True)
                ref = np.concatenate([np_walk(hp, ha, us[a:a + 256], by, *DEFAULTS[by]) for a in range(0, us.size, 256)])
                check_bound(s.cpu().numpy(), ref[inv, pairs[:, 1]], hp, DEFAULTS[by][0], f"fb-pages-food {by}")
            res = rank_scores(s, ds, ks)
            sc = s.cpu().numpy().astype(np.float64)
            if ds is rk:
                mrr, hits = np_rank(sc[:P // 51], sc[P // 51:].reshape(P // 51, 50), ks)
                assert abs(res["mrr"] - mrr) <= 1e-12 * mrr, (what, by)
                assert [res[f"hits@{k}"] for k in ks] == hits, (what, by)
            else:
                assert [res[f"hits@{k}"] for k in ks] == np_hits(sc, ds.y.reshape(-1)[0::2].cpu().numpy(), ks), (what, by)
    # recall@100 of the held-out partner: PPR reaches beyond two hops, so it retrieves at least what Adamic-Adar does
    E = tst.ei.shape[1]
    P = tst.y.shape[0] // 2
    pos = tst.pos1[E::2][:P][tst.y.reshape(-1)[0::2] > 0.5]
    ids_ppr, _ = recommend_global(tst, pos[:, 0].contiguous(), k=100, by="ppr")
    ids_aa, _ = recommend(tst, pos[:, 0].contiguous(), k=100, by="aa")
    rec_ppr = float((ids_ppr == pos[:, 1:2]).any(1).float().mean())
    rec_aa = float((ids_aa == pos[:, 1:2]).any(1).float().mean())
    assert rec_ppr >= rec_aa, (rec_ppr, rec_aa)
    # the candidate table of the PPR shortlist and the model's re-ranking of it
    src = pos[:200, 0].contiguous()
    ids, sc = recommend_global(tst, src, k=20, by="ppr")
    ds = D.candidate_dataset(bg, 2, src, ids)
    m = ids >= 0
    assert torch.equal(ds.cand_mask, m) and torch.equal(ds.cand_ids, ids)
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
    assert ops.GLOBAL_HEURISTICS == ("katz", "ppr")
