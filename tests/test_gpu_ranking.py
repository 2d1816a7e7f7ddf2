"""Ranking evaluation: hits@K against shared negatives (twowl_hits_at_k), MRR / hits@k against per-positive negatives
(twowl_rank_metrics), the filtered per-source negative sampler (twowl_tail_negative_sample), the ranking table
(TwoWL.operators.datasets.ranking_dataset) and TwoWL.model.train.test_ranking.

The metrics are checked against numpy restatements of OGB's evaluators (ogb/linkproppred/evaluate.py _eval_hits, _eval_mrr):
hits are integer counts over n_pos / P in double on both sides, so they must be EQUAL; MRR sums 1/rank in a different order, so
it is held to 1e-12 relative. The argument checks of the C ABI run without a GPU."""
import ctypes

import numpy as np
import pytest
import torch

from helpers import parity, state_dict_from
from oracle import twowl_oracle as O

EINVAL, ENOSPC = -22, -28


# ------------------------------------------------------------------------------ CPU: argument checks of the C ABI

@pytest.fixture(scope="module")
def L():
    import __graft_entry__ as ge
    ge._load_build_module().build()          # nvcc cross-compiles sm_100a without a GPU
    import twowl_b200._lib as lib_mod
    return lib_mod


def _ks(*v):
    return (ctypes.c_int64 * len(v))(*v)


FAKE = 256          # a non-null device address: every call below returns before it could be dereferenced


def _err(L, rc, code, text):
    assert rc == code, (rc, L.lib.twowl_last_error())
    assert text in L.lib.twowl_last_error().decode()


def test_hits_at_k_argument_errors(L):
    lib = L.lib
    nb = lib.twowl_hits_at_k_workspace_bytes(100)
    assert nb > lib.twowl_hits_at_k_workspace_bytes(0) > 0
    _err(L, lib.twowl_hits_at_k(FAKE, FAKE, -1, _ks(1), 1, FAKE, FAKE, nb, None), EINVAL, "n out of range")
    _err(L, lib.twowl_hits_at_k(FAKE, FAKE, 1 << 31, _ks(1), 1, FAKE, FAKE, nb, None), EINVAL, "n out of range")
    _err(L, lib.twowl_hits_at_k(None, FAKE, 100, _ks(1), 1, FAKE, FAKE, nb, None), EINVAL, "null pointer")
    _err(L, lib.twowl_hits_at_k(FAKE, FAKE, 100, _ks(1), 1, None, FAKE, nb, None), EINVAL, "null pointer")
    _err(L, lib.twowl_hits_at_k(FAKE, FAKE, 100, _ks(1), 0, FAKE, FAKE, nb, None), EINVAL, "ks must hold")
    _err(L, lib.twowl_hits_at_k(FAKE, FAKE, 100, _ks(*range(1, 18)), 17, FAKE, FAKE, nb, None), EINVAL, "ks must hold")
    _err(L, lib.twowl_hits_at_k(FAKE, FAKE, 100, _ks(5, 0), 2, FAKE, FAKE, nb, None), EINVAL, "ks must hold")
    _err(L, lib.twowl_hits_at_k(FAKE, FAKE, 100, None, 1, FAKE, FAKE, nb, None), EINVAL, "ks must hold")
    _err(L, lib.twowl_hits_at_k(FAKE, FAKE, 100, _ks(1, 50), 2, FAKE, FAKE, nb - 1, None), ENOSPC, "workspace too small")


def test_rank_metrics_argument_errors(L):
    lib = L.lib
    nb = lib.twowl_rank_metrics_workspace_bytes(1000)
    assert nb >= lib.twowl_rank_metrics_workspace_bytes(0) > 0
    _err(L, lib.twowl_rank_metrics(FAKE, FAKE, -1, 10, _ks(1), 1, FAKE, FAKE, nb, None), EINVAL, "bad sizes")
    _err(L, lib.twowl_rank_metrics(FAKE, FAKE, 1000, 0, _ks(1), 1, FAKE, FAKE, nb, None), EINVAL, "bad sizes")
    _err(L, lib.twowl_rank_metrics(FAKE, FAKE, 1 << 31, 10, _ks(1), 1, FAKE, FAKE, nb, None), EINVAL, "bad sizes")
    _err(L, lib.twowl_rank_metrics(FAKE, None, 1000, 10, _ks(1), 1, FAKE, FAKE, nb, None), EINVAL, "null pointer")
    _err(L, lib.twowl_rank_metrics(FAKE, FAKE, 1000, 10, _ks(1), 1, None, FAKE, nb, None), EINVAL, "null pointer")
    _err(L, lib.twowl_rank_metrics(FAKE, FAKE, 1000, 10, _ks(-3), 1, FAKE, FAKE, nb, None), EINVAL, "ks must hold")
    _err(L, lib.twowl_rank_metrics(FAKE, FAKE, 1000, 10, _ks(*range(1, 18)), 17, FAKE, FAKE, nb, None), EINVAL, "ks must hold")
    _err(L, lib.twowl_rank_metrics(FAKE, FAKE, 1000, 10, _ks(1, 3), 2, FAKE, FAKE, 0, None), ENOSPC, "workspace too small")


def test_tail_negative_sample_argument_errors(L):
    lib = L.lib
    f = lib.twowl_tail_negative_sample
    nb = lib.twowl_tail_negative_sample_workspace_bytes(1000, 100, 10)
    assert nb > lib.twowl_tail_negative_sample_workspace_bytes(1000, 0, 10) > 0
    _err(L, f(FAKE, 1, FAKE, 1, -1, 50, FAKE, 100, 10, 0, 16, FAKE, FAKE, FAKE, nb, None), EINVAL, "bad sizes")
    _err(L, f(FAKE, 1, FAKE, 1, 1000, 50, FAKE, 100, 0, 0, 16, FAKE, FAKE, FAKE, nb, None), EINVAL, "bad sizes")
    _err(L, f(FAKE, 1, FAKE, 1, 1000, 0, FAKE, 100, 10, 0, 16, FAKE, FAKE, FAKE, nb, None), EINVAL, "bad sizes")
    _err(L, f(FAKE, 1, FAKE, 1, 1000, 50, FAKE, 100, 10, 0, 0, FAKE, FAKE, FAKE, nb, None), EINVAL, "bad sizes")
    _err(L, f(FAKE, 1, FAKE, 1, 1000, 50, FAKE, 1 << 16, 1 << 15, 0, 16, FAKE, FAKE, FAKE, nb, None), EINVAL, "below 2^31")
    _err(L, f(FAKE, 1, FAKE, 1, 1000, 1 << 31, FAKE, 100, 10, 0, 16, FAKE, FAKE, FAKE, nb, None), EINVAL, "below 2^31")
    _err(L, f(FAKE, 1, FAKE, 1, 1000, 50, FAKE, 100, 10, 0, 16, FAKE, None, FAKE, nb, None), EINVAL, "null pointer")
    _err(L, f(FAKE, 1, FAKE, 1, 1000, 50, None, 100, 10, 0, 16, FAKE, FAKE, FAKE, nb, None), EINVAL, "null pointer")
    _err(L, f(FAKE, 1, FAKE, 1, 1000, 50, FAKE, 100, 10, 0, 16, None, FAKE, FAKE, nb, None), EINVAL, "null pointer")
    _err(L, f(None, 1, FAKE, 1, 1000, 50, FAKE, 100, 10, 0, 16, FAKE, FAKE, FAKE, nb, None), EINVAL, "null pointer")
    _err(L, f(FAKE, 1, FAKE, 1, 1000, 50, FAKE, 100, 10, 0, 16, FAKE, FAKE, FAKE, nb - 1, None), ENOSPC, "workspace too small")


def test_ranking_ops_refuse_cpu_tensors_and_bad_ks(L):
    from twowl_b200 import ops
    s, y = torch.zeros(4), torch.tensor([1.0, 0.0, 0.0, 0.0])
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.hits_at_k(s, y, [1])
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.rank_metrics(s, torch.zeros(4, 3), [1])
    e = torch.zeros(3, dtype=torch.int64)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.sample_tail_negatives(e, e, 5, e, 2)
    for bad in ([], [0], [1, -2], list(range(1, 18))):
        with pytest.raises(ValueError, match="ks must hold"):
            ops._rank_ks(bad)


# ------------------------------------------------------------------------------ GPU: metrics against numpy

def np_hits(score, label, ks):
    """OGB _eval_hits: kth = K-th largest negative, hits@K = #(pos > kth) / n_pos, 1.0 with fewer than K negatives."""
    score = np.asarray(score, dtype=np.float64)
    pos, neg = score[label > 0.5], score[~(label > 0.5)]
    if pos.size == 0 or np.isnan(score).any():
        return [float("nan")] * len(ks)
    srt = np.sort(neg)
    return [1.0 if neg.size < K else int((pos > srt[neg.size - K]).sum()) / pos.size for K in ks]


def np_rank(pos, neg, ks, chunk=8192):
    """OGB _eval_mrr: rank = 0.5 (#(neg > pos) + #(neg >= pos)) + 1 -> (MRR, [hits@k]), chunked over rows."""
    P = pos.shape[0]
    if P == 0 or np.isnan(pos).any() or np.isnan(neg).any():
        return float("nan"), [float("nan")] * len(ks)
    rank = np.empty(P)
    for a in range(0, P, chunk):
        p = pos[a:a + chunk, None]
        n = neg[a:a + chunk]
        rank[a:a + chunk] = 0.5 * ((n > p).sum(1) + (n >= p).sum(1)) + 1
    return float((1.0 / rank).mean()), [int((rank <= k).sum()) / P for k in ks]


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from twowl_b200 import ops as o
    return o


def _same(got, ref):
    """float lists equal, NaN matching NaN."""
    got, ref = np.asarray(got, dtype=np.float64), np.asarray(ref, dtype=np.float64)
    return got.shape == ref.shape and bool(np.all((got == ref) | (np.isnan(got) & np.isnan(ref))))


def _scores(rng, n, ties):
    s = rng.standard_normal(n).astype(np.float32)
    if ties:
        s = np.round(s, 1).astype(np.float32)     # ~60 distinct values
        z = rng.random(n) < 0.05
        s[z] = np.where(rng.random(int(z.sum())) < 0.5, np.float32(-0.0), np.float32(0.0))
    return s


@pytest.mark.gpu
@pytest.mark.parametrize("n_pos,n_neg,ties", [(1, 1, False), (1, 1, True), (3, 2, False), (7, 40, True), (500, 499, False),
                                              (1000, 20000, True), (20000, 300000, False), (200000, 3000000, True)])
def test_hits_at_k_matches_ogb(ops, n_pos, n_neg, ties):
    rng = np.random.default_rng(n_pos * 7 + n_neg + ties)
    score = _scores(rng, n_pos + n_neg, ties)
    label = np.zeros(n_pos + n_neg, dtype=np.float32)
    label[rng.permutation(n_pos + n_neg)[:n_pos]] = 1.0
    ks = sorted({1, 2, 3, 20, 50, 100, n_neg, n_neg + 1, 10 * n_neg + 7})[:16]
    got = ops.hits_at_k(torch.from_numpy(score).cuda(), torch.from_numpy(label).cuda(), ks).cpu().numpy()
    ref = np_hits(score, label, ks)
    assert _same(got[:len(ks)], ref), (list(zip(ks, got, ref)))
    assert got[len(ks)] == n_pos and got[len(ks) + 1] == n_neg
    assert got[ks.index(n_neg + 1)] == 1.0


@pytest.mark.gpu
def test_hits_at_k_zero_signs_tie(ops):
    # +0.0 and -0.0 are the same score: a positive at +0.0 is NOT above a negative at -0.0
    score = torch.tensor([0.0, -0.0, -0.0, 0.0, 1.0], device="cuda")
    label = torch.tensor([1.0, 1.0, 0.0, 0.0, 0.0], device="cuda")
    got = ops.hits_at_k(score, label, [1, 2, 3, 4]).cpu().tolist()
    assert got == [0.0, 0.0, 0.0, 1.0, 2.0, 3.0]


@pytest.mark.gpu
def test_hits_at_k_nan_and_no_positive(ops):
    rng = np.random.default_rng(5)
    score = rng.standard_normal(1000).astype(np.float32)
    label = (rng.random(1000) < 0.1).astype(np.float32)
    ks = [1, 10, 5000]
    for where in (np.flatnonzero(label > 0.5)[0], np.flatnonzero(label < 0.5)[0]):
        s = score.copy()
        s[where] = np.nan
        got = ops.hits_at_k(torch.from_numpy(s).cuda(), torch.from_numpy(label).cuda(), ks).cpu().numpy()
        assert np.isnan(got[:3]).all() and got[3] == label.sum() and got[4] == 1000 - label.sum()
    got = ops.hits_at_k(torch.from_numpy(score).cuda(), torch.zeros(1000, device="cuda"), ks).cpu().numpy()
    assert np.isnan(got[:3]).all() and got[3] == 0 and got[4] == 1000
    got = ops.hits_at_k(torch.zeros(0, device="cuda"), torch.zeros(0, device="cuda"), ks).cpu().numpy()
    assert np.isnan(got[:3]).all() and got[3] == 0 and got[4] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("P,k,ties", [(1, 1, False), (1, 1, True), (5, 3, True), (33, 31, False), (1000, 100, True),
                                      (4097, 257, False), (100000, 1000, True)])
def test_rank_metrics_matches_ogb(ops, P, k, ties):
    rng = np.random.default_rng(P + 13 * k + ties)
    pos = _scores(rng, P, ties)
    neg = _scores(rng, P * k, ties).reshape(P, k)
    ks = sorted({1, 3, 10, 20, 50, 100, k, k + 1})
    dp, dn = torch.from_numpy(pos).cuda(), torch.from_numpy(neg).cuda()
    got = ops.rank_metrics(dp, dn, ks)
    again = ops.rank_metrics(dp, dn, ks)
    assert torch.equal(got.view(torch.int64), again.view(torch.int64)), "two runs differ"
    got = got.cpu().numpy()
    mrr, hits = np_rank(pos, neg, ks)
    assert abs(got[0] - mrr) <= 1e-12 * abs(mrr), (got[0], mrr)
    assert _same(got[1:1 + len(ks)], hits), list(zip(ks, got[1:], hits))
    assert got[-1] == P


@pytest.mark.gpu
def test_rank_metrics_nan_and_empty(ops):
    rng = np.random.default_rng(9)
    pos = torch.from_numpy(rng.standard_normal(64).astype(np.float32)).cuda()
    neg = torch.from_numpy(rng.standard_normal((64, 10)).astype(np.float32)).cuda()
    for t, at in ((pos, (7,)), (neg, (63, 9))):
        keep = t[at].item()
        t[at] = float("nan")
        got = ops.rank_metrics(pos, neg, [1, 5]).cpu().numpy()
        t[at] = keep
        assert np.isnan(got[:3]).all() and got[3] == 64
    got = ops.rank_metrics(torch.zeros(0, device="cuda"), torch.zeros((0, 4), device="cuda"), [1]).cpu().numpy()
    assert np.isnan(got[:2]).all() and got[2] == 0
    # rank by hand: negatives (3, 1, 1) around a positive at 1 -> opt 1, pess 3 -> rank 3
    got = ops.rank_metrics(torch.tensor([1.0], device="cuda"), torch.tensor([[3.0, 1.0, 1.0]], device="cuda"), [2, 3]).cpu()
    assert got.tolist() == [1.0 / 3.0, 0.0, 1.0, 1.0]


# ------------------------------------------------------------------------------ GPU: per-source negatives

def _check_tail(out, src, n, edges):
    """every entry in [0, n), not its source, not an excluded edge in either direction; rows distinct."""
    out, src = out.cpu().numpy(), src.cpu().numpy()
    assert out.min() >= 0 and out.max() < n
    assert not (out == src[:, None]).any()
    ekeys = np.unique(np.concatenate([edges[0] * n + edges[1], edges[1] * n + edges[0]]))
    assert not np.isin(src[:, None] * n + out, ekeys).any()
    srt = np.sort(out, axis=1)
    assert (np.diff(srt, axis=1) != 0).all(), "a row repeats a node"


@pytest.mark.gpu
@pytest.mark.parametrize("n,m,P,k", [(50, 200, 30, 5), (2000, 20000, 500, 50), (1 << 16, 1 << 19, 20000, 100)])
def test_tail_sampler_contract(ops, n, m, P, k):
    rng = np.random.default_rng(n + m)
    edges = rng.integers(0, n, size=(2, m))                 # duplicates and self loops included
    src = rng.integers(0, n, size=P)
    e, s = torch.from_numpy(edges).cuda(), torch.from_numpy(src).cuda()
    out = ops.sample_tail_negatives(e[0], e[1], n, s, k, seed=7)
    assert out.shape == (P, k) and out.dtype == torch.int64
    _check_tail(out, s, n, edges)
    assert torch.equal(out, ops.sample_tail_negatives(e[0], e[1], n, s, k, seed=7))
    assert not torch.equal(out, ops.sample_tail_negatives(e[0], e[1], n, s, k, seed=8))
    et = torch.from_numpy(np.ascontiguousarray(edges.T)).cuda()        # strided edge columns
    assert torch.equal(out, ops.sample_tail_negatives(et[:, 0], et[:, 1], n, s, k, seed=7))
    torch.manual_seed(3)
    a = ops.sample_tail_negatives(e[0], e[1], n, s, k)
    torch.manual_seed(3)
    assert torch.equal(a, ops.sample_tail_negatives(e[0], e[1], n, s, k))


@pytest.mark.gpu
def test_tail_sampler_hub_graph(ops):
    n = 300
    spokes = np.arange(1, 250)
    edges = np.stack([np.zeros_like(spokes), spokes])        # hub 0: 50 allowed nodes (250..299)
    edges = np.concatenate([edges, np.stack([spokes[:-1], spokes[1:]])], axis=1)
    src = np.concatenate([[0, 0, 0], np.random.default_rng(0).integers(1, n, size=200)])
    e, s = torch.from_numpy(edges).cuda(), torch.from_numpy(src).cuda()
    out = ops.sample_tail_negatives(e[0], e[1], n, s, 20, seed=1, rounds=256)
    _check_tail(out, s, n, edges)
    assert bool((out[:3] >= 250).all())
    full = ops.sample_tail_negatives(e[0], e[1], n, s[:1], 50, seed=1, rounds=4096)   # every allowed node of the hub
    assert sorted(full[0].tolist()) == list(range(250, 300))
    with pytest.raises(ValueError, match="fewer than k=51 allowed"):
        ops.sample_tail_negatives(e[0], e[1], n, s, 51, seed=1, rounds=64)
    with pytest.raises(ValueError, match="unfilled"):
        ops.sample_tail_negatives(e[0], e[1], n, torch.tensor([n], device="cuda"), 1, seed=1)


@pytest.mark.gpu
def test_tail_sampler_is_uniform(ops):
    """Each row is a uniform k-subset of the allowed nodes, so every allowed node appears equally often per source: chi-square over
    the counts of 40000 rows of one source on a 16-node graph (seeded, so deterministic), against a loose fixed bound."""
    n, reps, k = 16, 40000, 3
    edges = np.array([[0, 0, 0, 5, 2, 9], [1, 2, 7, 0, 3, 9]])      # source 0 excludes 1, 2, 5, 7 (and itself)
    allowed = np.array([w for w in range(n) if w not in (0, 1, 2, 5, 7)])
    e = torch.from_numpy(edges).cuda()
    src = torch.zeros(reps, dtype=torch.int64, device="cuda")
    out = ops.sample_tail_negatives(e[0], e[1], n, src, k, seed=11).cpu().numpy()
    cnt = np.bincount(out.reshape(-1), minlength=n)
    assert cnt[np.setdiff1d(np.arange(n), allowed)].sum() == 0
    exp = reps * k / allowed.size
    chi2 = float((((cnt[allowed] - exp) ** 2) / exp).sum())
    assert chi2 < 40.0, (chi2, cnt)                           # 10 degrees of freedom: P(chi2 > 40) ~ 2e-5


# ------------------------------------------------------------------------------ GPU: end to end on fb-pages-food

CFG1 = dict(channels_1wl=64, channels_2wl=24, depth1=2, depth2=2, dp_lin0=0., dp_lin1=0., dp_emb=0., dp_1wl0=0.,
            dp_2wl=0., dp_1wl1=0., act0=True, act1=True)


@pytest.fixture(scope="module")
def fbg(fb):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import TwoWL.model.model as model
    import TwoWL.operators.datasets as D
    n = int(fb["num_nodes"][0])
    ep, en = (torch.from_numpy(fb[k].astype(np.int64)).cuda() for k in ("edge_pos", "edge_neg"))
    bg = D.BaseGraph(torch.zeros((n, 0), device="cuda"), None, ep, en, torch.from_numpy(fb["num_pos"]),
                     torch.from_numpy(fb["num_neg"]), "2wl_l")
    bg.preprocess()
    bg.setPosDegreeFeature()
    sd = state_dict_from(fb)
    mod = model.LocalWLNet(sd["emb.0.weight"].shape[0] - 1, False, None, **CFG1)
    mod.load_state_dict(sd, strict=True)
    return D, bg, mod.cuda().eval(), sd


def _logits(mod, ds):
    idx = ds.ei.shape[1] + torch.arange(ds.y.shape[0], device="cuda")
    with torch.no_grad():
        return mod(ds.x, ds.ei, ds.pos1, idx, ds.ei2, True).reshape(-1), idx


@pytest.mark.gpu
def test_ranking_dataset_layout(fbg):
    D, bg, _, _ = fbg
    n, k = bg.num_nodes, 50
    ds = D.ranking_dataset(bg, 2, num_neg=k)
    assert ds.rank_k == k and ds.x is bg.x[2] and ds.ei is bg.edge_indexs[2]
    npos = [int(v) for v in bg.num_pos]
    pos = bg.edge_pos[:, bg.edge_pos.shape[1] - npos[2]:][:, 0::2]
    P = pos.shape[1]
    E = ds.ei.shape[1]
    assert ds.pos1.shape == (E + 2 * P * (1 + k), 2) and ds.y.shape == (2 * P * (1 + k), 1)
    assert torch.equal(ds.pos1[:E], ds.ei.t())
    pred = ds.pos1[E:]
    assert torch.equal(pred[0::2], pred[1::2].flip(1))                           # double(): (a, b) then (b, a)
    und = pred[0::2]
    assert torch.equal(und[:P], pos.t())
    neg = und[P:].reshape(P, k, 2)
    assert torch.equal(neg[:, :, 0], pos[0][:, None].expand(P, k))               # sources = the positives' u
    ep = bg.edge_pos.cpu().numpy()
    _check_tail(neg[:, :, 1], pos[0], n, ep)                                      # filtered against every split's positives
    assert bool((ds.y[:2 * P] == 1).all()) and bool((ds.y[2 * P:] == 0).all())
    ref = O.get_ei2(n, ds.ei.cpu().numpy(), pred.t().cpu().numpy())
    assert np.array_equal(ds.ei2.cpu().numpy(), ref)
    again = D.ranking_dataset(bg, 2, num_neg=k)
    assert torch.equal(again.pos1, ds.pos1)                                       # seed=0 by default
    assert not torch.equal(D.ranking_dataset(bg, 2, num_neg=k, seed=1).pos1, ds.pos1)
    imp = D.ranking_dataset(bg, 1, num_neg=3, pattern="2wl_l_implicit")
    assert np.array_equal(imp.ei2.materialize().cpu().numpy(), D.ranking_dataset(bg, 1, num_neg=3).ei2.cpu().numpy())
    for bad in (0, 3):
        with pytest.raises(ValueError, match="split"):
            D.ranking_dataset(bg, bad, num_neg=k)


@pytest.mark.gpu
def test_ranking_end_to_end_fb_pages_food(fbg):
    from TwoWL.model.train import test_ranking
    D, bg, mod, sd = fbg
    k = 50
    ds = D.ranking_dataset(bg, 2, num_neg=k)
    out, idx = _logits(mod, ds)
    args = (ds.x.cpu(), ds.ei.cpu(), ds.pos1.cpu(), idx.cpu(), ds.ei2.cpu().numpy())
    with torch.no_grad():
        o32 = O.local_wl_forward(sd, *args)
        o64 = O.local_wl_forward({kk: v.double() for kk, v in sd.items()}, *args)
    parity(out, o32.reshape(-1), o64.reshape(-1), "ranking table logits")
    out2, _ = _logits(mod, ds)
    assert torch.equal(out, out2), "the eval forward is not bitwise repeatable"
    ks = (1, 10, 20, 50, 51)
    res = test_ranking(mod, ds, ks)
    lg = out.cpu().numpy().astype(np.float64)
    P = lg.size // (1 + k)
    mrr, hits = np_rank(lg[:P], lg[P:].reshape(P, k), ks)
    assert set(res) == {"mrr"} | {f"hits@{kk}" for kk in ks}
    assert abs(res["mrr"] - mrr) <= 1e-12 * mrr and 0 < mrr <= 1
    assert [res[f"hits@{kk}"] for kk in ks] == hits and hits[-1] == 1.0

    # the existing test split: hits@K of its positives against the shared negatives
    tst = D.dataset(*bg.split(2))
    res = test_ranking(mod, tst, (1, 5, 20, 50, 100000))
    out, _ = _logits(mod, tst)
    lab = tst.y.reshape(-1)[0::2].cpu().numpy()
    ref = np_hits(out.cpu().numpy(), lab, (1, 5, 20, 50, 100000))
    assert [res[f"hits@{kk}"] for kk in (1, 5, 20, 50, 100000)] == ref and ref[-1] == 1.0
