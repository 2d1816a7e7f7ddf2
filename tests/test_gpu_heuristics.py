"""Neighbourhood link-prediction heuristics: the simple adjacency (twowl_simple_adjacency), the pair scores cn / jaccard / aa / ra
(twowl_link_plan + twowl_link_heuristics), TwoWL.model.train.heuristic_scores and rank_scores.

The references are numpy / scipy.sparse float64 restatements of the definitions:
  N(x) = {y != x : (x, y) or (y, x) is an edge}, d(x) = |N(x)|, c = |N(u) ∩ N(v)|,
  cn = c, jaccard = c / (d(u) + d(v) - c) (0 when that is 0), aa = sum 1 / ln d(w) (0 for d(w) <= 1), ra = sum 1 / d(w).
cn is an integer and jaccard the fp32 quotient of two exact integers, so both must be EQUAL. aa and ra are double sums rounded
once to fp32: they must lie within 0.5 ulp32(ref) + 2 c 2^-53 ref of the float64 reference (the final rounding, plus the
rounding of c double terms and their sum). The argument checks of the C ABI run without a GPU."""
import ctypes

import numpy as np
import pytest
import scipy.sparse as sp
import torch

EINVAL, ENOSPC = -22, -28
FAKE = 256          # a non-null device address: every call below returns before it could be dereferenced
HEUR_LONG, HEUR_CHUNK = 64, 64   # TWOWL_HEUR_LONG / TWOWL_HEUR_CHUNK of include/twowl.h


# ------------------------------------------------------------------------------ CPU: argument checks of the C ABI

@pytest.fixture(scope="module")
def L():
    import __graft_entry__ as ge
    ge._load_build_module().build()          # nvcc cross-compiles sm_100a without a GPU
    import twowl_b200._lib as lib_mod
    return lib_mod


def _err(L, rc, code, text):
    assert rc == code, (rc, L.lib.twowl_last_error())
    assert text in L.lib.twowl_last_error().decode()


def test_simple_adjacency_argument_errors(L):
    lib = L.lib
    f = lib.twowl_simple_adjacency
    nb = lib.twowl_simple_adjacency_workspace_bytes(1000)
    assert nb > lib.twowl_simple_adjacency_workspace_bytes(0) > 0
    _err(L, f(FAKE, 1, FAKE, 1, -1, 50, FAKE, FAKE, FAKE, FAKE, nb, None), EINVAL, "bad sizes")
    _err(L, f(FAKE, 1, FAKE, 1, 1 << 30, 50, FAKE, FAKE, FAKE, FAKE, nb, None), EINVAL, "bad sizes")
    _err(L, f(FAKE, 1, FAKE, 1, 1000, -1, FAKE, FAKE, FAKE, FAKE, nb, None), EINVAL, "bad sizes")
    _err(L, f(FAKE, 1, FAKE, 1, 1000, (1 << 31) - 1, FAKE, FAKE, FAKE, FAKE, nb, None), EINVAL, "bad sizes")
    _err(L, f(None, 1, FAKE, 1, 1000, 50, FAKE, FAKE, FAKE, FAKE, nb, None), EINVAL, "null pointer")
    _err(L, f(FAKE, 1, None, 1, 1000, 50, FAKE, FAKE, FAKE, FAKE, nb, None), EINVAL, "null pointer")
    _err(L, f(FAKE, 1, FAKE, 1, 1000, 50, None, FAKE, FAKE, FAKE, nb, None), EINVAL, "null pointer")
    _err(L, f(FAKE, 1, FAKE, 1, 1000, 50, FAKE, None, FAKE, FAKE, nb, None), EINVAL, "null pointer")
    _err(L, f(FAKE, 1, FAKE, 1, 1000, 50, FAKE, FAKE, None, FAKE, nb, None), EINVAL, "null pointer")
    _err(L, f(FAKE, 1, FAKE, 1, 1000, 50, FAKE, FAKE, FAKE, FAKE, nb - 1, None), ENOSPC, "workspace too small")


def test_link_plan_argument_errors(L):
    lib = L.lib
    f = lib.twowl_link_plan
    nb = lib.twowl_link_plan_workspace_bytes(1000)
    assert nb >= lib.twowl_link_plan_workspace_bytes(0) > 0
    _err(L, f(FAKE, 50, FAKE, 1, FAKE, 1, -1, FAKE, FAKE, FAKE, nb, None), EINVAL, "bad sizes")
    _err(L, f(FAKE, 50, FAKE, 1, FAKE, 1, 1 << 31, FAKE, FAKE, FAKE, nb, None), EINVAL, "bad sizes")
    _err(L, f(FAKE, -1, FAKE, 1, FAKE, 1, 1000, FAKE, FAKE, FAKE, nb, None), EINVAL, "bad sizes")
    _err(L, f(None, 50, FAKE, 1, FAKE, 1, 1000, FAKE, FAKE, FAKE, nb, None), EINVAL, "null pointer")
    _err(L, f(FAKE, 50, None, 1, FAKE, 1, 1000, FAKE, FAKE, FAKE, nb, None), EINVAL, "null pointer")
    _err(L, f(FAKE, 50, FAKE, 1, None, 1, 1000, FAKE, FAKE, FAKE, nb, None), EINVAL, "null pointer")
    _err(L, f(FAKE, 50, FAKE, 1, FAKE, 1, 1000, None, FAKE, FAKE, nb, None), EINVAL, "null pointer")
    _err(L, f(FAKE, 50, FAKE, 1, FAKE, 1, 1000, FAKE, None, FAKE, nb, None), EINVAL, "null pointer")
    _err(L, f(FAKE, 50, FAKE, 1, FAKE, 1, 1000, FAKE, FAKE, FAKE, nb - 1, None), ENOSPC, "workspace too small")


def test_link_heuristics_argument_errors(L):
    lib = L.lib
    f = lib.twowl_link_heuristics
    nb = lib.twowl_link_heuristics_workspace_bytes(100)
    assert nb > lib.twowl_link_heuristics_workspace_bytes(0) > 0
    _err(L, f(FAKE, FAKE, 50, FAKE, 1, FAKE, 1, -1, FAKE, 100, FAKE, FAKE, nb, None), EINVAL, "bad sizes")
    _err(L, f(FAKE, FAKE, 50, FAKE, 1, FAKE, 1, 1 << 31, FAKE, 100, FAKE, FAKE, nb, None), EINVAL, "bad sizes")
    _err(L, f(FAKE, FAKE, 50, FAKE, 1, FAKE, 1, 1000, FAKE, -1, FAKE, FAKE, nb, None), EINVAL, "bad sizes")
    _err(L, f(FAKE, FAKE, -1, FAKE, 1, FAKE, 1, 1000, FAKE, 100, FAKE, FAKE, nb, None), EINVAL, "bad sizes")
    _err(L, f(None, FAKE, 50, FAKE, 1, FAKE, 1, 1000, FAKE, 100, FAKE, FAKE, nb, None), EINVAL, "null pointer")
    _err(L, f(FAKE, FAKE, 50, None, 1, FAKE, 1, 1000, FAKE, 100, FAKE, FAKE, nb, None), EINVAL, "null pointer")
    _err(L, f(FAKE, FAKE, 50, FAKE, 1, FAKE, 1, 1000, None, 100, FAKE, FAKE, nb, None), EINVAL, "null pointer")
    _err(L, f(FAKE, FAKE, 50, FAKE, 1, FAKE, 1, 1000, FAKE, 100, None, FAKE, nb, None), EINVAL, "null pointer")
    _err(L, f(FAKE, FAKE, 50, FAKE, 1, FAKE, 1, 1000, FAKE, 100, FAKE, FAKE, nb - 1, None), ENOSPC, "workspace too small")


def test_heuristic_ops_refuse_cpu_tensors(L):
    from twowl_b200 import ops
    e = torch.zeros(3, dtype=torch.int64)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.simple_adjacency(e, e, 5)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.link_heuristics(torch.zeros(6, dtype=torch.int64), torch.zeros(0, dtype=torch.int32), e, e)
    assert ops.HEURISTICS == ("cn", "jaccard", "aa", "ra")


# ------------------------------------------------------------------------------ numpy / scipy restatement

def np_adjacency(row, col, n):
    """-> (ptr, adj): np.unique of the symmetrised, loop-free keys row * n + col."""
    row, col = np.asarray(row, np.int64), np.asarray(col, np.int64)
    keep = row != col
    r, c = row[keep], col[keep]
    keys = np.unique(np.concatenate((r * n + c, c * n + r)))
    ptr = np.searchsorted(keys // n, np.arange(n + 1), side="left").astype(np.int64) if n else np.zeros(1, np.int64)
    return ptr, (keys % n).astype(np.int32)


def np_heuristics(ptr, adj, u, v):
    """float64 (cn, jaccard as fp32, aa, ra) of the pairs (u, v) over a simple adjacency (ptr, adj)."""
    n = ptr.size - 1
    A = sp.csr_matrix((np.ones(adj.size), adj.astype(np.int64), ptr), shape=(n, n))
    d = np.diff(ptr).astype(np.float64)
    with np.errstate(divide="ignore"):
        w_aa = np.where(d > 1, 1.0 / np.log(np.maximum(d, 2)), 0.0)
        w_ra = np.where(d > 0, 1.0 / np.maximum(d, 1), 0.0)
    common = A[u].multiply(A[v]).tocsr()
    cn = np.asarray(common.sum(axis=1)).reshape(-1)
    aa = common @ w_aa
    ra = common @ w_ra
    den = d[u] + d[v] - cn
    with np.errstate(divide="ignore", invalid="ignore"):
        jac = np.where(den > 0, np.float32(cn) / np.float32(den), np.float32(0)).astype(np.float32)
    return cn, jac, aa, ra


def check_scores(got, ref, what):
    """got: fp32 [4, P] (torch); ref: np_heuristics."""
    g = got.cpu().numpy()
    cn, jac, aa, ra = ref
    assert np.array_equal(g[0], cn.astype(np.float32)), f"{what}: cn differs"
    assert np.array_equal(g[1], jac), f"{what}: jaccard differs from the fp32 quotient"
    for row, r, name in ((2, aa, "aa"), (3, ra, "ra")):
        tol = 0.5 * np.spacing(np.abs(r).astype(np.float32)).astype(np.float64) + 2 * cn * 2.0 ** -53 * np.abs(r)
        err = np.abs(g[row].astype(np.float64) - r)
        bad = err > tol
        assert not bad.any(), f"{what}: {name} off by {err[bad][:5]} > {tol[bad][:5]} at {np.nonzero(bad)[0][:5]}"


# ------------------------------------------------------------------------------ GPU

@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from twowl_b200 import ops as o
    return o


def cu(a, dtype=torch.int64):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dtype).cuda()


@pytest.mark.gpu
def test_simple_adjacency_matches_numpy(ops):
    rng = np.random.default_rng(0)
    n, m = 3000, 40000          # ids drawn below 2500: nodes 2500..2999 are isolated, num_nodes > max id + 1
    r, c = rng.integers(0, 2500, m), rng.integers(0, 2500, m)
    r = np.concatenate((r, r[:5000], np.arange(300)))                 # duplicates and self loops
    c = np.concatenate((c, c[:5000], np.arange(300)))
    r, c = np.concatenate((r, c[:2000])), np.concatenate((c, r[:2000]))   # some edges given in both directions, the rest in one
    ptr, adj = ops.simple_adjacency(cu(r), cu(c), n)
    rp, ra = np_adjacency(r, c, n)
    assert ptr.dtype == torch.int64 and adj.dtype == torch.int32
    assert np.array_equal(ptr.cpu().numpy(), rp) and np.array_equal(adj.cpu().numpy(), ra)
    assert int(ptr[-1]) == adj.numel() and int((ptr[2501:] - ptr[2500:-1]).abs().sum()) == 0
    # a transposed view of a [E, 2] tensor (strides 2) gives the same adjacency
    ec = cu(np.stack((r, c), axis=1))
    p2, a2 = ops.simple_adjacency(ec[:, 0], ec[:, 1], n)
    assert torch.equal(p2, ptr) and torch.equal(a2, adj)
    p0, a0 = ops.simple_adjacency(cu(np.zeros(0)), cu(np.zeros(0)), 7)
    assert torch.equal(p0.cpu(), torch.zeros(8, dtype=torch.int64)) and a0.numel() == 0
    e0 = ops.link_heuristics(p0, a0, cu([0, 3, 6]), cu([0, 5, 6]))       # no edges at all: every score is 0
    assert torch.equal(e0, torch.zeros(4, 3, device="cuda"))
    for bad in (-1, n):
        rb = r.copy()
        rb[17] = bad
        with pytest.raises(ValueError, match="outside"):
            ops.simple_adjacency(cu(rb), cu(c), n)
    torch.cuda.synchronize()


def _queries(rng, n, ptr, P):
    """P random pairs plus u == v, isolated endpoints and repeats."""
    deg = np.diff(ptr)
    iso = np.nonzero(deg == 0)[0]
    hub = np.argsort(deg)[-32:]
    u, v = rng.integers(0, n, P), rng.integers(0, n, P)
    k = P // 10
    v[:k] = u[:k]                                           # u == v
    if iso.size:
        u[k:2 * k] = rng.choice(iso, k)                     # isolated endpoint
        u[2 * k:2 * k + 10], v[2 * k:2 * k + 10] = iso[0], iso[-1]
    u[3 * k:4 * k], v[3 * k:4 * k] = rng.choice(hub, k), rng.choice(hub, k)   # hub pairs
    u[4 * k:5 * k], v[4 * k:5 * k] = u[5 * k:6 * k], v[5 * k:6 * k]           # repeated pairs
    return u, v


def _check_graph(ops, r, c, n, P, seed, what):
    rng = np.random.default_rng(seed)
    ptr, adj = ops.simple_adjacency(cu(r), cu(c), n)
    hp, ha = ptr.cpu().numpy(), adj.cpu().numpy()
    u, v = _queries(rng, n, hp, P)
    tu, tv = cu(u), cu(v)
    got = ops.link_heuristics(ptr, adj, tu, tv)
    assert got.shape == (4, P) and got.dtype == torch.float32
    check_scores(got, np_heuristics(hp, ha, u, v), what)
    assert torch.equal(got, ops.link_heuristics(ptr, adj, tu, tv)), f"{what}: not bitwise repeatable"
    sw = ops.link_heuristics(ptr, adj, tv, tu)
    assert torch.equal(got.view(torch.int32), sw.view(torch.int32)), f"{what}: score(u, v) != score(v, u) bitwise"
    return hp


@pytest.mark.gpu
def test_scores_erdos_renyi(ops):
    rng = np.random.default_rng(1)
    n, m = 20000, 300000
    r, c = rng.integers(0, n - 500, m), rng.integers(0, n - 500, m)    # the last 500 nodes are isolated
    _check_graph(ops, r, c, n, 150_000, 2, "Erdos-Renyi")


@pytest.mark.gpu
def test_scores_rmat_with_hubs(ops):
    from TwoWL.operators.synthetic import rmat_edges
    s, d, n = rmat_edges(16, 1_000_000, (0.57, 0.19, 0.19, 0.05), 3, torch.device("cuda"))
    hp = _check_graph(ops, s.cpu().numpy(), d.cpu().numpy(), n, 150_000, 4, "R-MAT")
    assert np.diff(hp).max() > 20 * HEUR_LONG       # the hubs' pairs take the chunked path


def _plan_chunks(ops, ptr, u, v):
    """(bad ids, chunks, probes) of twowl_link_plan for these pairs."""
    from twowl_b200._lib import lib
    P = u.numel()
    off = torch.empty(P + 1, dtype=torch.int64, device="cuda")
    info = torch.empty(3, dtype=torch.int64, device="cuda")
    nb = lib.twowl_link_plan_workspace_bytes(P)
    ws = torch.empty(nb, dtype=torch.uint8, device="cuda")
    assert lib.twowl_link_plan(ptr.data_ptr(), ptr.numel() - 1, u.data_ptr(), 1, v.data_ptr(), 1, P, off.data_ptr(),
                               info.data_ptr(), ws.data_ptr(), nb, torch.cuda.current_stream().cuda_stream) == 0
    return info.tolist()


@pytest.mark.gpu
def test_hub_pairs_take_the_chunked_path(ops):
    """Hubs 0 and 1 have 50 000 neighbours each, 40 000 of them shared (nodes 2 .. 40 001), plus a background graph among the
    small nodes so that d(w) varies. A hub-hub pair probes min(d) = 50 000 entries (50 001 with the hub-hub edge) >
    TWOWL_HEUR_LONG = 64, so it is cut into ceil(50 001 / 64) = 782 chunks of TWOWL_HEUR_CHUNK = 64 probes; the plan's chunk
    count below proves the chunked path runs. Pairs of a hub with a small node stay on the short path."""
    rng = np.random.default_rng(5)
    n = 120_000
    shared = np.arange(2, 40_002)
    only0, only1 = np.arange(40_002, 50_002), np.arange(50_002, 60_002)
    r = np.concatenate(([0], np.zeros(shared.size + only0.size, np.int64), np.ones(shared.size + only1.size, np.int64),
                        rng.integers(2, n, 400_000)))
    c = np.concatenate(([1], shared, only0, shared, only1, rng.integers(2, n, 400_000)))
    ptr, adj = ops.simple_adjacency(cu(r), cu(c), n)
    hp, ha = ptr.cpu().numpy(), adj.cpu().numpy()
    assert hp[1] - hp[0] == 50_001 and hp[2] - hp[1] == 50_001
    small = rng.integers(2, n, 2000)
    u = np.concatenate(([0, 1, 0, 1], np.zeros(1000, np.int64), small[:1000], np.full(64, 0)))
    v = np.concatenate(([1, 0, 0, 1], small[:1000], np.ones(1000, np.int64), np.full(64, 1)))
    tu, tv = cu(u), cu(v)
    bad, chunks, probes = _plan_chunks(ops, ptr, tu, tv)
    hubhub = 2 + 2 + 64                                       # (0,1), (1,0), (0,0), (1,1) and 64 repeats of (0, 1)
    assert bad == 0 and chunks == hubhub * -(-50_001 // HEUR_CHUNK)
    got = ops.link_heuristics(ptr, adj, tu, tv)
    check_scores(got, np_heuristics(hp, ha, u, v), "hub pairs")
    assert int(got[0, 0]) == 40_000 and float(got[1, 2]) == 1.0
    assert torch.equal(got, ops.link_heuristics(ptr, adj, tu, tv))
    assert torch.equal(got.view(torch.int32), ops.link_heuristics(ptr, adj, tv, tu).view(torch.int32))
    assert torch.equal(got[:, 0:1].expand(4, 64), got[:, -64:])


@pytest.mark.gpu
def test_bad_query_id_raises_index_error(ops):
    rng = np.random.default_rng(6)
    n = 500
    ptr, adj = ops.simple_adjacency(cu(rng.integers(0, n, 3000)), cu(rng.integers(0, n, 3000)), n)
    u, v = cu(rng.integers(0, n, 100)), cu(rng.integers(0, n, 100))
    for bad in (-1, n, 1 << 40):
        ub = u.clone()
        ub[7] = bad
        with pytest.raises(IndexError, match="outside"):
            ops.link_heuristics(ptr, adj, ub, v)
        with pytest.raises(IndexError, match="outside"):
            ops.link_heuristics(ptr, adj, u, ub)
    torch.cuda.synchronize()                                   # the device is still healthy
    assert ops.link_heuristics(ptr, adj, u, v).isfinite().all()
    assert ops.link_heuristics(ptr, adj, u[:0], v[:0]).shape == (4, 0)


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
def test_heuristics_end_to_end_fb_pages_food(fbg):
    from test_gpu_ranking import np_hits, np_rank
    from TwoWL.model.train import heuristic_scores, rank_scores, test_ranking
    from twowl_b200 import ops
    D, bg, mod = fbg
    n = bg.num_nodes
    tst = D.dataset(*bg.split(2))
    rk = D.ranking_dataset(bg, 2, num_neg=50)
    ks = (1, 10, 20, 50, 100)
    for ds, what in ((tst, "test split"), (rk, "ranking table")):
        E = ds.ei.shape[1]
        P = ds.y.shape[0] // 2
        h = heuristic_scores(ds)
        assert list(h) == list(ops.HEURISTICS) and all(t.shape == (P,) and t.dtype == torch.float32 for t in h.values())
        ei = ds.ei.cpu().numpy()
        hp, ha = np_adjacency(ei[0], ei[1], n)
        pairs = ds.pos1[E::2].cpu().numpy()
        check_scores(torch.stack([h[k] for k in ops.HEURISTICS]), np_heuristics(hp, ha, pairs[:, 0], pairs[:, 1]), what)
        for name, s in h.items():
            res = rank_scores(s, ds, ks)
            sc = s.cpu().numpy().astype(np.float64)
            if ds is rk:
                mrr, hits = np_rank(sc[:P // 51], sc[P // 51:].reshape(P // 51, 50), ks)
                assert abs(res["mrr"] - mrr) <= 1e-12 * mrr, (what, name)
                assert [res[f"hits@{k}"] for k in ks] == hits, (what, name)
            else:
                ref = np_hits(sc, ds.y.reshape(-1)[0::2].cpu().numpy(), ks)
                assert [res[f"hits@{k}"] for k in ks] == ref, (what, name)
        # the model's logits ranked by rank_scores == test_ranking, bit for bit
        idx = E + torch.arange(ds.y.shape[0], device="cuda")
        with torch.no_grad():
            logits = mod(ds.x, ds.ei, ds.pos1, idx, ds.ei2, True)
        assert rank_scores(logits, ds, ks) == test_ranking(mod, ds, ks)
    from twowl_b200 import graph
    assert graph.simple_adjacency(tst.ei, n) is graph.simple_adjacency(tst.ei, n)   # built once per edge tensor
