"""BUDDY on the device: the subgraph sketches (twowl_sketch_init / _hop, ops.link_sketches), the pair features
(twowl_sketch_pair_features, ops.sketch_features), TwoWL.model.buddy.BUDDY and train.buddy_fit / buddy_scores.

The sketches are compared bit for bit with a numpy restatement: the hash in uint64 arithmetic, the hops as np.minimum.reduceat /
np.maximum.reduceat over the CSR, masked edges deleted by scipy. The features are compared with a float64 numpy restatement of
the estimators over the device's own sketches: Z and J are exact, so only the double log and the final rounding can differ. The
estimates are held against exact neighbourhood counts from scipy boolean powers of A + I, and BUDDY against a float64 torch
restatement (BatchNorm1d in training mode) that loads the same state_dict.
"""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

from test_gpu_heuristics import FAKE, EINVAL, ENOSPC, L, _err, cu, np_adjacency  # noqa: F401  (L is a fixture)
from test_gpu_ncn import _rel_err, deleted_graph
from test_gpu_recommend import fbg  # noqa: F401  (a fixture: fb-pages-food's graph and the reference model)
from test_gpu_seal import _rmat

# ------------------------------------------------------------------------------ CPU: argument checks


def test_sketch_argument_errors(L):
    lib = L.lib
    init = lib.twowl_sketch_init
    for n, npm, p in ((-1, 128, 8), ((1 << 31) - 1, 128, 8)):
        _err(L, init(n, npm, p, 0, FAKE, FAKE, None), EINVAL, "bad sizes")
    for npm, p in ((100, 8), (0, 8), (2048, 8), (16, 8), (128, 3), (128, 11)):
        _err(L, init(10, npm, p, 0, FAKE, FAKE, None), EINVAL, "num_perm")
    _err(L, init(10, 128, 8, 0, None, FAKE, None), EINVAL, "null pointer")
    _err(L, init(10, 128, 8, 0, FAKE, None, None), EINVAL, "null pointer")
    _err(L, init(10, 128, 8, 0, FAKE + 4, FAKE, None), EINVAL, "16-byte aligned")

    nb = lib.twowl_sketch_hop_workspace_bytes(1000, 128, 8, 64)
    assert nb > lib.twowl_sketch_hop_workspace_bytes(1000, 128, 8, 1 << 20) > 0
    assert lib.twowl_sketch_hop_workspace_bytes(1000, 100, 8, 64) == 0
    hop = lib.twowl_sketch_hop

    def h(n=50, nnz=1000, npm=128, p=8, chunk=64, ptr=FAKE, adj=FAKE, mi=FAKE, hi=FAKE, mo=2 * FAKE, ho=2 * FAKE, ws=FAKE, wsb=nb):
        return hop(ptr, adj, n, nnz, None, npm, p, chunk, mi, hi, mo, ho, ws, wsb, None)

    for kw in (dict(n=-1), dict(n=(1 << 31) - 1), dict(nnz=-1), dict(nnz=1 << 31)):
        _err(L, h(**kw), EINVAL, "bad sizes")
    for kw in (dict(npm=96 + 8), dict(npm=1056), dict(p=12), dict(p=2)):
        _err(L, h(**kw), EINVAL, "num_perm")
    for kw in (dict(chunk=0), dict(chunk=-5), dict(chunk=(1 << 30) + 1)):
        _err(L, h(**kw), EINVAL, "chunk")
    for kw in ("ptr", "adj", "mi", "hi", "mo", "ho"):
        _err(L, h(**{kw: None}), EINVAL, "null pointer")
    _err(L, h(mo=FAKE), EINVAL, "different rows")
    _err(L, h(hi=FAKE + 8), EINVAL, "16-byte aligned")
    _err(L, h(wsb=nb - 1), ENOSPC, "workspace too small")
    _err(L, h(ws=None), EINVAL, "null pointer")

    feat = lib.twowl_sketch_pair_features

    def f(k=2, n=50, npm=128, p=8, mh=FAKE, hll=FAKE, u=FAKE, v=FAKE, P=10, out=FAKE, info=FAKE):
        return feat(k, n, npm, p, mh, hll, u, 1, v, 1, P, out, info, None)

    for k in (0, 4, -1):
        _err(L, f(k=k), EINVAL, "hops")
    for kw in (dict(n=-1), dict(P=-1), dict(P=1 << 31)):
        _err(L, f(**kw), EINVAL, "bad sizes")
    for kw in (dict(npm=48), dict(p=11)):
        _err(L, f(**kw), EINVAL, "num_perm")
    for kw in ("mh", "hll", "u", "v", "out", "info"):
        _err(L, f(**{kw: None}), EINVAL, "null pointer")


def test_buddy_ops_refuse_cpu_tensors_and_bad_arguments(L):
    from twowl_b200 import ops
    ptr, adj, s = torch.zeros(6, dtype=torch.int64), torch.zeros(0, dtype=torch.int32), torch.zeros(3, dtype=torch.int64)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.link_sketches(ptr, adj)
    sk = ops.LinkSketches(torch.zeros((3, 5, 128), dtype=torch.int32), torch.zeros((3, 5, 256), dtype=torch.uint8), 2, 128, 8, 0)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.sketch_features(sk, s, s)
    if torch.cuda.is_available():
        ptr, adj = ptr.cuda(), adj.cuda()
        for kw in (dict(hops=0), dict(hops=4), dict(num_perm=100), dict(hll_p=3), dict(chunk=0)):
            with pytest.raises(ValueError):
                ops.link_sketches(ptr, adj, **kw)


def test_buddy_parameter_names(L):
    from TwoWL.model.buddy import BUDDY
    keys = set(BUDDY(2).state_dict())
    bn = {f"bn_labels.{k}" for k in ("weight", "bias", "running_mean", "running_var", "num_batches_tracked")}
    assert keys == {"label_lin_layer.weight", "label_lin_layer.bias", "lin.weight", "lin.bias"} | bn
    m = BUDDY(3, node_feat_dim=6, hidden=16)
    assert m.label_lin_layer.weight.shape == (15, 15) and m.lin_feat.weight.shape == (16, 24) and m.lin.weight.shape == (1, 31)
    with pytest.raises(ValueError, match="multiple of 4"):
        BUDDY(2, hidden=10)
    with pytest.raises(ValueError, match="hops"):
        BUDDY(4)


# ------------------------------------------------------------------------------ numpy restatements

_GOLD = 0x9E3779B97F4A7C15


def np_hash(seed: int, idx) -> np.ndarray:
    """common.cuh's hash_u32 (splitmix64 finaliser) in uint64 arithmetic."""
    with np.errstate(over="ignore"):
        z = np.asarray(idx, np.uint64) + np.uint64((seed * _GOLD + _GOLD) % 2 ** 64)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return (z >> np.uint64(32)).astype(np.uint32)


def np_init(n, num_perm, p, seed):
    """Hop-0 sketches of include/twowl.h: seed_mh = 2 seed, seed_hll = 2 seed + 1."""
    s_mh, s_hll = (2 * seed) % 2 ** 64, (2 * seed + 1) % 2 ** 64
    j, u = np.meshgrid(np.arange(num_perm, dtype=np.uint64), np.arange(n, dtype=np.uint64))
    mh = np_hash(s_mh, (j << np.uint64(32)) | u)
    m = 1 << p
    h = np_hash(s_hll, np.arange(n, dtype=np.uint64)).astype(np.int64)
    reg, w = h & (m - 1), h >> p
    bitlen = np.frexp(w.astype(np.float64))[1]                 # bit length of w (0 for w = 0)
    rank = np.where(w > 0, (32 - bitlen) - p + 1, 33 - p)
    hll = np.zeros((n, m), np.uint8)
    hll[np.arange(n), reg] = rank
    return mh, hll


def np_hop(hp, ha, prev, op):
    """One propagation step over the CSR (hp, ha): op (np.minimum / np.maximum) of a row with its neighbours' rows."""
    n = hp.size - 1
    out = prev.copy()
    cnt = np.diff(hp)
    nz = cnt > 0
    if ha.size:
        red = op.reduceat(prev[ha], hp[:-1][nz], axis=0)
        out[nz] = op(out[nz], red)
    return out


def np_sketches(hp, ha, hops, num_perm, p, seed):
    mh, hll = np_init(hp.size - 1, num_perm, p, seed)
    mhs, hlls = [mh], [hll]
    for _ in range(hops):
        mhs.append(np_hop(hp, ha, mhs[-1], np.minimum))
        hlls.append(np_hop(hp, ha, hlls[-1], np.maximum))
    return np.stack(mhs), np.stack(hlls)


_HLL_THRESHOLD = {4: 10.0, 5: 20.0, 6: 40.0, 7: 80.0, 8: 220.0, 9: 400.0, 10: 900.0}


def np_est(M):
    """HyperLogLog estimate of register rows M (uint8 [..., m]) in float64, as include/twowl.h states it."""
    m = M.shape[-1]
    p = m.bit_length() - 1
    md = float(m)
    Z = np.ldexp(1.0, -M.astype(np.int64)).sum(-1)            # exact: dyadic terms >= 2^-33
    V = (M == 0).sum(-1)
    alpha = {16: 0.673, 32: 0.697, 64: 0.709}.get(m, 0.7213 / (1.0 + 1.079 / md))
    E = alpha * md * md / Z
    with np.errstate(divide="ignore"):
        lc = md * np.log(md / V.astype(np.float64))
    return np.where((V > 0) & (lc <= _HLL_THRESHOLD[p]), lc, E)


def np_features(mh, hll, u, v, k):
    """float64 restatement of twowl_sketch_pair_features over given sketches -> (fp32 [P, k^2 + 2k], the float64 values before the
    clamp and the rounding, the largest estimate of each row)."""
    mh = mh.view(np.uint32)
    P, npm = len(u), mh.shape[2]
    eu = np.stack([np_est(hll[d][u]) for d in range(k + 1)], 1)
    ev = np.stack([np_est(hll[d][v]) for d in range(k + 1)], 1)
    I = np.zeros((P, k + 1, k + 1))
    for d1 in range(1, k + 1):
        for d2 in range(1, k + 1):
            J = (mh[d1][u] == mh[d2][v]).sum(-1) / float(npm)
            I[:, d1, d2] = J * np_est(np.maximum(hll[d1][u], hll[d2][v]))
    A = (I[:, 1:, 1:] + I[:, :-1, :-1]) - (I[:, :-1, 1:] + I[:, 1:, :-1])
    cols = [A[:, a, b] for a in range(k) for b in range(k)]
    for d in range(1, k + 1):
        s = np.zeros(P)
        for d2 in range(k):
            s = s + A[:, d - 1, d2]
        cols.append((eu[:, d] - eu[:, d - 1]) - s)
    for d in range(1, k + 1):
        s = np.zeros(P)
        for d1 in range(k):
            s = s + A[:, d1, d - 1]
        cols.append((ev[:, d] - ev[:, d - 1]) - s)
    raw = np.stack(cols, 1) if P else np.zeros((0, k * k + 2 * k))
    scale = np.maximum(eu.max(1, initial=0.0), ev.max(1, initial=0.0)) if P else np.zeros(0)
    return np.maximum(raw, 0.0).astype(np.float32), raw, scale


def check_features(got, mh, hll, u, v, k, what):
    """Within one fp32 ulp of the float64 restatement; where a difference of two estimates cancels, also within the double log's
    rounding (2^-50 of the row's largest estimate), the only operation that may round differently."""
    ref, raw, scale = np_features(mh, hll, u, v, k)
    g = got.cpu().numpy()
    assert g.shape == ref.shape, what
    tol = np.spacing(np.abs(ref)) + 2.0 ** -50 * scale[:, None]
    bad = np.abs(g.astype(np.float64) - ref.astype(np.float64)) > tol
    assert not bad.any(), f"{what}: {int(bad.sum())} features off, e.g. {g[bad][:4]} vs {ref[bad][:4]}"


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from twowl_b200 import ops as o
    return o


def _graphs():
    rng = np.random.default_rng(11)
    er = (rng.integers(0, 300, 1500), rng.integers(0, 300, 1500), 400)                 # 300..399 isolated
    rr, rc = _rmat(10, 8000, rng)
    hub_r = np.concatenate([np.zeros(3000, np.int64), rng.integers(1, 4000, 4000)])     # node 0: degree 3000
    hub_c = np.concatenate([np.arange(1, 3001), rng.integers(1, 4000, 4000)])
    return {"er": er, "rmat": (rr, rc, 1024), "hub": (hub_r, hub_c, 4100)}


def _sk_np(sk):
    return sk.minhash.cpu().numpy(), sk.hll.cpu().numpy()


# ------------------------------------------------------------------------------ sketches, bit for bit

@pytest.mark.gpu
@pytest.mark.parametrize("name", ["er", "rmat", "hub"])
@pytest.mark.parametrize("hops", [1, 2, 3])
def test_sketches_match_numpy(ops, name, hops):
    r, c, n = _graphs()[name]
    ptr, adj = ops.simple_adjacency(cu(r), cu(c), n)
    hp, ha = ptr.cpu().numpy(), adj.cpu().numpy()
    if name == "hub":
        assert np.diff(hp).max() >= 3000
    num_perm, p = (128, 8) if hops != 3 else (64, 5)
    sk = ops.link_sketches(ptr, adj, hops, num_perm, p, seed=5)
    mh, hll = np_sketches(hp, ha, hops, num_perm, p, 5)
    assert sk.minhash.shape == (hops + 1, n, num_perm) and sk.minhash.dtype == torch.int32
    assert sk.hll.shape == (hops + 1, n, 1 << p) and sk.hll.dtype == torch.uint8
    gm, gh = _sk_np(sk)
    assert np.array_equal(gm.view(np.uint32), mh), f"{name} minhash"
    assert np.array_equal(gh, hll), f"{name} hll"
    deg = np.diff(hp)
    for d in range(hops + 1):                                  # isolated nodes keep their hop-0 sketch
        assert np.array_equal(gm[d][deg == 0], gm[0][deg == 0]) and np.array_equal(gh[d][deg == 0], gh[0][deg == 0])


@pytest.mark.gpu
@pytest.mark.parametrize("num_perm,p", [(32, 4), (96, 7), (1024, 10)])
def test_sketch_widths(ops, num_perm, p):
    r, c, n = _graphs()["rmat"]
    ptr, adj = ops.simple_adjacency(cu(r), cu(c), n)
    sk = ops.link_sketches(ptr, adj, 2, num_perm, p, seed=3)
    mh, hll = np_sketches(ptr.cpu().numpy(), adj.cpu().numpy(), 2, num_perm, p, 3)
    gm, gh = _sk_np(sk)
    assert np.array_equal(gm.view(np.uint32), mh) and np.array_equal(gh, hll)


@pytest.mark.gpu
def test_sketches_independent_of_the_cut(ops):
    r, c, n = _graphs()["hub"]
    ptr, adj = ops.simple_adjacency(cu(r), cu(c), n)
    ref = ops.link_sketches(ptr, adj, 2, seed=1)
    for chunk in (1, 7, 64, 1000, 2999, 3000, 1 << 30):
        sk = ops.link_sketches(ptr, adj, 2, seed=1, chunk=chunk)
        assert torch.equal(sk.minhash, ref.minhash) and torch.equal(sk.hll, ref.hll), chunk
    again = ops.link_sketches(ptr, adj, 2, seed=1)
    assert torch.equal(again.minhash, ref.minhash) and torch.equal(again.hll, ref.hll)
    other = ops.link_sketches(ptr, adj, 2, seed=2)
    assert not torch.equal(other.minhash, ref.minhash)


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["rmat", "hub"])
def test_masked_sketches_match_deleted_graph(ops, name):
    r, c, n = _graphs()[name]
    ptr, adj = ops.simple_adjacency(cu(r), cu(c), n)
    hp, ha = ptr.cpu().numpy(), adj.cpu().numpy()
    rng = np.random.default_rng(9)
    e = rng.integers(0, ha.size, 400)
    rows = np.searchsorted(hp, e, side="right") - 1
    edges = np.stack([rows, ha[e]], 1)
    edges[::2] = edges[::2, ::-1]                                                        # both orientations
    dele = np.concatenate([edges, edges[:20], rng.integers(0, n, (40, 2)), [[3, 3]]])    # duplicates, non-edges, u == v
    mask = ops.adjacency_pair_mask(ptr, adj, cu(dele[:, 0]), cu(dele[:, 1]))
    dp, da = deleted_graph(hp, ha, dele)
    for chunk in (5, 64):
        got = ops.link_sketches(ptr, adj, 3, 64, 6, seed=2, entry_mask=mask, chunk=chunk)
        ref = ops.link_sketches(cu(dp), cu(da, torch.int32), 3, 64, 6, seed=2)
        assert torch.equal(got.minhash, ref.minhash) and torch.equal(got.hll, ref.hll), chunk
    mh, hll = np_sketches(dp, da, 3, 64, 6, 2)
    assert np.array_equal(got.minhash.cpu().numpy().view(np.uint32), mh) and np.array_equal(got.hll.cpu().numpy(), hll)


# ------------------------------------------------------------------------------ features

def _pairs(hp, ha, n, rng, P):
    e = rng.integers(0, ha.size, P // 2)
    rows = np.searchsorted(hp, e, side="right") - 1
    u = np.concatenate([rows, rng.integers(0, n, P - P // 2)])
    v = np.concatenate([ha[e], rng.integers(0, n, P - P // 2)])
    return u, v


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["er", "rmat", "hub"])
@pytest.mark.parametrize("hops,num_perm,p", [(1, 128, 8), (2, 128, 8), (3, 64, 4), (2, 1024, 10)])
def test_features_match_float64(ops, name, hops, num_perm, p):
    r, c, n = _graphs()[name]
    ptr, adj = ops.simple_adjacency(cu(r), cu(c), n)
    hp, ha = ptr.cpu().numpy(), adj.cpu().numpy()
    u, v = _pairs(hp, ha, n, np.random.default_rng(4), 600)
    deg = np.diff(hp)
    iso, hub = np.flatnonzero(deg == 0), int(np.argmax(deg))
    extra = [(5, 5), (hub, hub), (hub, 1)] + ([(int(iso[0]), 3), (int(iso[0]), int(iso[1]))] if iso.size > 1 else [])
    u, v = np.concatenate([u, [a for a, _ in extra]]), np.concatenate([v, [b for _, b in extra]])
    sk = ops.link_sketches(ptr, adj, hops, num_perm, p, seed=7)
    f = ops.sketch_features(sk, cu(u), cu(v))
    assert f.shape == (len(u), hops * hops + 2 * hops) and f.dtype == torch.float32
    mh, hll = _sk_np(sk)
    check_features(f, mh, hll, u, v, hops, name)
    # (v, u): A transposed, B_u and B_v swapped, bit for bit
    g = ops.sketch_features(sk, cu(v), cu(u))
    k = hops
    A, At = f[:, :k * k].reshape(-1, k, k), g[:, :k * k].reshape(-1, k, k)
    assert torch.equal(A, At.transpose(1, 2))
    assert torch.equal(f[:, k * k:k * k + k], g[:, k * k + k:]) and torch.equal(f[:, k * k + k:], g[:, k * k:k * k + k])
    assert torch.equal(f, ops.sketch_features(sk, cu(u), cu(v)))


@pytest.mark.gpu
def test_features_edge_cases(ops):
    r, c, n = _graphs()["er"]
    ptr, adj = ops.simple_adjacency(cu(r), cu(c), n)
    sk = ops.link_sketches(ptr, adj, 2)
    assert ops.sketch_features(sk, cu([]), cu([])).shape == (0, 8)
    iso = ops.sketch_features(sk, cu([350, 350]), cu([360, 350])).cpu().numpy()        # isolated endpoints: nothing beyond hop 0
    mh, hll = _sk_np(sk)
    check_features(torch.from_numpy(iso), mh, hll, np.array([350, 350]), np.array([360, 350]), 2, "isolated")
    assert np.all(iso[:, [1, 2, 3]] == 0) and np.all(iso[:, 5] == 0) and np.all(iso[:, 7] == 0)
    for bu, bv in (([0, n], [1, 2]), ([-1], [1]), ([1], [n + 5])):
        with pytest.raises(IndexError):
            ops.sketch_features(sk, cu(bu), cu(bv))
    p0, a0 = ops.simple_adjacency(cu([]), cu([]), 9)                                    # no edges at all
    e0 = ops.link_sketches(p0, a0, 3)
    assert torch.equal(e0.minhash[3], e0.minhash[0]) and torch.equal(e0.hll[3], e0.hll[0])
    f0 = ops.sketch_features(e0, cu([0, 3, 8]), cu([0, 5, 8]))
    mh, hll = _sk_np(e0)
    check_features(f0, mh, hll, np.array([0, 3, 8]), np.array([0, 5, 8]), 3, "empty graph")
    z = ops.link_sketches(torch.zeros(1, dtype=torch.int64, device="cuda"), torch.zeros(0, dtype=torch.int32, device="cuda"), 2)
    assert z.minhash.shape == (3, 0, 128)
    with pytest.raises(IndexError):
        ops.sketch_features(z, cu([0]), cu([0]))


# ------------------------------------------------------------------------------ statistical agreement with exact counts

@pytest.mark.gpu
def test_estimates_agree_with_exact_counts(ops):
    rng = np.random.default_rng(21)
    n, m_edges = 3000, 7500
    r, c = rng.integers(0, n, m_edges), rng.integers(0, n, m_edges)
    ptr, adj = ops.simple_adjacency(cu(r), cu(c), n)
    hp, ha = ptr.cpu().numpy(), adj.cpu().numpy()
    k, num_perm, p = 3, 1024, 10
    m = 1 << p
    sk = ops.link_sketches(ptr, adj, k, num_perm, p, seed=13)
    A = sp.csr_matrix((np.ones(ha.size), ha.astype(np.int64), hp), shape=(n, n)) + sp.identity(n, format="csr")
    R = [sp.identity(n, format="csr")]
    for _ in range(k):
        R.append(((R[-1] @ A) > 0).astype(np.float64).tocsr())
    # cardinalities: every node's N_{<=d}, d = 1..3
    _, hll = _sk_np(sk)
    size = np.stack([np.asarray(R[d].sum(1)).ravel() for d in range(1, k + 1)])
    est = np.stack([np_est(hll[d]) for d in range(1, k + 1)])
    big = size >= 50
    rel = np.abs(est[big] - size[big]) / size[big]
    sigma = 1.04 / np.sqrt(m)
    assert big.sum() >= 1000
    assert np.median(rel) <= sigma, np.median(rel)
    assert np.mean(rel <= 4 * sigma) >= 0.99, np.mean(rel <= 4 * sigma)
    # intersections I(d1, d2) = J U over >= 10^3 pairs of neighbours and two-hop pairs
    u, v = _pairs(hp, ha, n, rng, 3000)
    f_pairs = ops.sketch_features(sk, cu(u), cu(v))             # runs the device estimator on the same pairs
    mh = sk.minhash.cpu().numpy().view(np.uint32)
    errs, bounds = [], []
    for d1 in range(1, k + 1):
        for d2 in range(1, k + 1):
            inter = np.asarray(R[d1][u].multiply(R[d2][v]).sum(1)).ravel()
            union = np.asarray(R[d1][u].maximum(R[d2][v]).sum(1)).ravel()
            J_hat = (mh[d1][u] == mh[d2][v]).sum(-1) / num_perm
            I_hat = J_hat * np_est(np.maximum(hll[d1][u], hll[d2][v]))
            sel = inter >= 20
            J = inter[sel] / union[sel]
            errs.append(np.abs(I_hat[sel] - inter[sel]) / inter[sel])
            # relative standard error of J from num_perm draws, plus HyperLogLog's 1.04 / sqrt(m) for the union
            bounds.append(np.sqrt((1 - J) / (J * num_perm)) + sigma)
    errs, bounds = np.concatenate(errs), np.concatenate(bounds)
    assert errs.size >= 1000, errs.size
    # E|Z| = 0.80 sigma for a normal error; the bound allows 1.25 times the mean standard error
    assert errs.mean() <= 1.25 * bounds.mean(), (errs.mean(), bounds.mean())
    assert torch.isfinite(f_pairs).all()


# ------------------------------------------------------------------------------ BUDDY against a float64 restatement

def _buddy_batch(ops, hops=2):
    """A doubled edge tensor, a batch of positives and negatives, and the features and graph buddy_fit hands the model for it."""
    from TwoWL.utils import double, sample_block
    r, c, n = _graphs()["rmat"]
    hp, ha = np_adjacency(r, c, n)
    rows = np.repeat(np.arange(n), np.diff(hp))
    und = np.stack([rows, ha], 1)[rows < ha]
    ei = cu(np.stack([und, und[:, ::-1]], 1).reshape(-1, 2).T)
    rng = np.random.default_rng(8)
    pos_ids = np.sort(rng.choice(und.shape[0], 40, replace=False))
    neg = rng.integers(0, n, (30, 2))
    pairs = np.concatenate([und[pos_ids], neg[neg[:, 0] != neg[:, 1]]])
    ptr, adj = ops.simple_adjacency(ei[0], ei[1], n)
    mask = ops.adjacency_pair_mask(ptr, adj, cu(und[pos_ids, 0]), cu(und[pos_ids, 1]))
    sf = ops.sketch_features(ops.link_sketches(ptr, adj, hops, entry_mask=mask), cu(pairs[:, 0]), cu(pairs[:, 1]))
    ei_new, _, _ = sample_block(double(cu(pos_ids), for_index=True), n, ei, None)
    keep = np.ones(ei.shape[1], bool)
    keep[2 * pos_ids], keep[2 * pos_ids + 1] = False, False
    return dict(n=n, ei=ei.cpu().numpy(), keep=keep, pairs=pairs, sf=sf, ei_new=ei_new)


def ref_buddy(mod, b, feat, training=True, bn_state=None):
    """float64 BUDDY on the CPU from mod's state_dict -> (logits, {name: leaf parameter}, the BatchNorm1d it ran)."""
    from oracle import twowl_oracle as O
    sd = {k: v.detach().cpu().double() for k, v in mod.state_dict().items()}
    P = {name: sd[name].clone().requires_grad_() for name, _ in mod.named_parameters()}
    bn = torch.nn.BatchNorm1d(mod.dim).double()
    with torch.no_grad():
        bn.weight.copy_(P["bn_labels.weight"])
        bn.bias.copy_(P["bn_labels.bias"])
        src = bn_state or sd
        bn.running_mean.copy_(src["bn_labels.running_mean"])
        bn.running_var.copy_(src["bn_labels.running_var"])
    bn.train(training)
    s = b["sf"].cpu().double() @ P["label_lin_layer.weight"].t() + P["label_lin_layer.bias"]
    s = torch.relu(torch.nn.functional.batch_norm(s, bn.running_mean, bn.running_var, P["bn_labels.weight"], P["bn_labels.bias"],
                                                  training, bn.momentum, bn.eps))
    x = s
    if feat is not None:
        ei = torch.from_numpy(b["ei"][:, b["keep"]])
        h = feat.cpu().double()
        eye = torch.eye(h.shape[1], dtype=torch.float64)
        hs = [h]
        for _ in range(mod.hops):
            hs.append(O.gcn_conv(hs[-1], ei, eye, torch.zeros(h.shape[1], dtype=torch.float64)))
        u, v = (torch.from_numpy(b["pairs"][:, k]) for k in (0, 1))
        hp = torch.cat([t[u] * t[v] for t in hs], 1)
        x = torch.cat((s, torch.relu(hp @ P["lin_feat.weight"].t() + P["lin_feat.bias"])), 1)
    return x @ P["lin.weight"].t() + P["lin.bias"], P, bn


# the NCN bound: ||got - ref|| <= BUDDY_REL ||ref|| per tensor
BUDDY_REL = 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("F", [0, 6])
def test_buddy_against_float64_restatement(ops, F):
    from TwoWL.model.buddy import BUDDY
    b = _buddy_batch(ops)
    torch.manual_seed(0)
    mod = BUDDY(2, dropout=0.0, node_feat_dim=F, hidden=16).cuda().train()
    feat = torch.randn((b["n"], F)).cuda() if F else None
    xs = mod.propagate(feat, b["ei_new"]) if F else None
    w = torch.randn((b["pairs"].shape[0], 1))
    before = {k: v.clone() for k, v in mod.state_dict().items()}
    out = mod(b["sf"], cu(b["pairs"]), xs)
    (out * w.cuda()).sum().backward()
    mod.load_state_dict(before)                                # the reference starts from the same running statistics
    o64, P, _ = ref_buddy(mod, b, feat)
    (o64 * w.double()).sum().backward()
    assert _rel_err(out, o64) <= BUDDY_REL, ("logits", _rel_err(out, o64))
    grads = {name: p.grad for name, p in mod.named_parameters()}
    assert set(grads) == set(P)
    for name, g in grads.items():
        if name == "label_lin_layer.bias":
            # training-mode BatchNorm subtracts the batch mean, so this gradient is zero up to rounding on both sides
            scale = float(P["label_lin_layer.weight"].grad.norm())
            assert float(g.norm()) <= 1e-5 * scale and float(P[name].grad.norm()) <= 1e-5 * scale
            continue
        assert _rel_err(g, P[name].grad) <= BUDDY_REL, (name, _rel_err(g, P[name].grad))
        # the check can fail: a halved or zeroed gradient is rejected
        assert _rel_err(0.5 * g, P[name].grad) > BUDDY_REL and _rel_err(0 * g, P[name].grad) > BUDDY_REL, name


@pytest.mark.gpu
def test_buddy_running_statistics_and_eval(ops):
    from TwoWL.model.buddy import BUDDY
    torch.manual_seed(1)
    mod = BUDDY(3, dropout=0.0).cuda().train()
    bn64 = None
    batches = [_buddy_batch(ops, hops=3)]
    g = torch.Generator().manual_seed(3)
    for i in range(2):                                          # three different batches: rows shuffled and subsampled
        idx = torch.randperm(batches[0]["pairs"].shape[0], generator=g)[: 50 - 10 * i]
        bb = dict(batches[0])
        bb["sf"], bb["pairs"] = batches[0]["sf"][idx.cuda()], batches[0]["pairs"][idx.numpy()]
        batches.append(bb)
    state = {k: v.detach().cpu().double() for k, v in mod.state_dict().items()}
    for bb in batches:
        with torch.no_grad():
            mod(bb["sf"])
        _, _, bn64 = ref_buddy(mod, bb, None, True, state)
        state = {"bn_labels.running_mean": bn64.running_mean.clone(), "bn_labels.running_var": bn64.running_var.clone()}
    rm, rv = mod.bn_labels.running_mean.cpu().double(), mod.bn_labels.running_var.cpu().double()
    assert int(mod.bn_labels.num_batches_tracked) == 3
    assert torch.allclose(rm, bn64.running_mean, rtol=1e-5, atol=1e-6 * float(bn64.running_mean.abs().max())), (rm, bn64.running_mean)
    assert torch.allclose(rv, bn64.running_var, rtol=1e-5, atol=0.0), (rv, bn64.running_var)
    mod.eval()
    with torch.no_grad():
        out = mod(batches[0]["sf"])
    o64, _, _ = ref_buddy(mod, batches[0], None, training=False)
    assert _rel_err(out, o64) <= BUDDY_REL, _rel_err(out, o64)


@pytest.mark.gpu
def test_buddy_dropout_repeatable(ops):
    from TwoWL.model.buddy import BUDDY
    b = _buddy_batch(ops)
    torch.manual_seed(0)
    feat = torch.randn((b["n"], 6)).cuda()
    mod = BUDDY(2, dropout=0.5, node_feat_dim=6, hidden=16).cuda().train()
    xs = mod.propagate(feat, b["ei_new"])
    pairs = cu(b["pairs"])
    res = []
    for _ in range(2):
        mod.zero_grad()
        out = mod(b["sf"], pairs, xs, seed=12345)
        out.sum().backward()
        res.append([out.detach().clone()] + [p.grad.clone() for p in mod.parameters()])
    assert all(torch.equal(x, y) for x, y in zip(*res))
    mod.zero_grad()
    assert not torch.equal(mod(b["sf"], pairs, xs, seed=777).detach(), res[0][0])


# ------------------------------------------------------------------------------ training, scores, re-ranking

@pytest.mark.gpu
def test_buddy_fit_repeatable_and_scores_batch_independent(fbg):
    from TwoWL.model.train import buddy_fit, buddy_scores
    D, bg, _ = fbg
    trn, tst = D.dataset(*bg.split(0)), D.dataset(*bg.split(2))
    runs = [buddy_fit(trn, 1, 256, seed=4) for _ in range(2)]
    (m0, l0), (m1, l1) = runs
    assert torch.equal(l0, l1) and l0.numel() > 0 and bool(torch.isfinite(l0).all())
    for (k0, a), (k1, b) in zip(m0.state_dict().items(), m1.state_dict().items()):
        assert k0 == k1 and torch.equal(a, b), k0
    s = buddy_scores(m0, tst)
    assert s.shape == (tst.y.shape[0] // 2,) and s.dtype == torch.float32 and bool(torch.isfinite(s).all())
    assert torch.equal(s, buddy_scores(m0, tst, batch_size=37))


@pytest.mark.gpu
def test_buddy_training_features_follow_the_protocol(fbg):
    """The features of a training batch equal those of the graph with the batch's positive edges deleted by scipy."""
    from TwoWL.model.train import _buddy_batch_features, _link_targets
    from twowl_b200 import graph, ops
    D, bg, _ = fbg
    trn = D.dataset(*bg.split(0))
    N = trn.x.shape[0]
    ptr, adj = graph.simple_adjacency(trn.ei, N)
    pairs, _ = _link_targets(trn)
    n_pos = trn.ei.shape[1] // 2
    gen = torch.Generator(device="cpu").manual_seed(4)
    ids = torch.randperm(pairs.shape[0], generator=gen)[:256].cuda()
    args = dict(num_perm=128, hll_p=8, seed=4)
    sf, pos = _buddy_batch_features(ptr, adj, pairs, ids, n_pos, 2, args)
    assert pos.numel() > 0
    hp, ha = ptr.cpu().numpy(), adj.cpu().numpy()
    dp, da = deleted_graph(hp, ha, pairs[pos].cpu().numpy())
    assert da.size == ha.size - 2 * pos.numel()
    ref = ops.sketch_features(ops.link_sketches(cu(dp), cu(da, torch.int32), 2, **args), pairs[ids, 0], pairs[ids, 1])
    assert torch.equal(sf, ref)
    kept = ops.sketch_features(ops.link_sketches(ptr, adj, 2, **args), pairs[ids, 0], pairs[ids, 1])
    assert not torch.equal(sf, kept)                            # the deletion changes what the positives see


@pytest.mark.gpu
def test_buddy_reranks_candidates(fbg):
    from TwoWL.model.train import buddy_fit, buddy_scores, recommend, rerank_scores
    D, bg, _ = fbg
    tst = D.dataset(*bg.split(2))
    E, P = tst.ei.shape[1], tst.y.shape[0] // 2
    src = tst.pos1[E::2][:P][tst.y.reshape(-1)[0::2] > 0.5][:100, 0].contiguous()
    ids, _ = recommend(tst, src, k=20, by="aa")
    ds = D.candidate_dataset(bg, 2, src, ids)
    mod, _ = buddy_fit(D.dataset(*bg.split(0)), 1, 256)
    nid, nlog = rerank_scores(buddy_scores(mod, ds), ds)
    assert torch.equal(torch.sort(nid, 1).values, torch.sort(ids, 1).values)
    assert bool((nlog[:, :-1] >= nlog[:, 1:]).all()) and bool(((nid < 0) == torch.isinf(nlog)).all())


# a sanity floor, not a claim: the measured numbers are in the README's BUDDY paragraph
BUDDY_FB = dict(epochs=40, batch_size=256, lr=5e-3, seed=0)
AUC_FLOOR = 0.80


@pytest.mark.gpu
def test_buddy_end_to_end_fb_pages_food(fbg):
    import time
    from TwoWL.model.train import buddy_fit, buddy_scores, rank_scores
    from twowl_b200 import ops
    D, bg, _ = fbg
    trn, tst = D.dataset(*bg.split(0)), D.dataset(*bg.split(2))
    labels = tst.y.reshape(-1)[0::2]
    t0 = time.perf_counter()
    mod, losses = buddy_fit(trn, **BUDDY_FB)
    torch.cuda.synchronize()
    secs = time.perf_counter() - t0
    s = buddy_scores(mod, tst)
    auc = float(ops.auc(s, labels)[0])
    rk = rank_scores(s, tst, (20, 50, 100))
    print(f"buddy training {secs:.2f} s, {losses.numel()} steps, loss {float(losses[0]):.4f} -> {float(losses[-1]):.4f}")
    print(f"fb-pages-food test buddy: AUC {auc:.4f} " + " ".join(f"{k} {v:.4f}" for k, v in rk.items()))
    assert losses[-1] < losses[0]
    assert auc > AUC_FLOOR, auc
