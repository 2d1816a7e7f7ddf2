"""GPU parity of the individual C-ABI kernels (through the Python operator layer) against the CPU
oracle and the reference-generated golden fixtures. Integer/index work is compared BIT-EXACT;
floating point within |a-b| <= 1e-6 + 1e-5*|b| (north_star tolerance) against an fp64 evaluation.
Run on a B200 box:  python -m pytest tests -m gpu -q
"""
import numpy as np
import pytest
import torch

from helpers import assert_close, fb_split, r32, sha
from oracle import twowl_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def U():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import TwoWL.utils as utils
    return utils


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def same(t, ref):
    t = t.detach().cpu().numpy()
    ref = np.asarray(ref)
    return t.shape == ref.shape and np.array_equal(t, ref)


# ------------------------------------------------------------------------------ golden vectors

def test_three_node_golden(U, golden):
    g = golden("three_node.npz")
    pos, pred = dev(g["pos"]), dev(g["pred"])
    assert same(U.double(dev(np.array([[0, 1], [1, 2]]))), g["pos"])
    assert same(U.double(dev(np.array([0, 2])), for_index=True), g["double_index"])
    ei2 = U.get_ei2(3, pos, pred)
    assert ei2.dtype == torch.int64 and not ei2.is_contiguous()  # cat(...).t() view, like utils.py:45
    assert same(ei2, g["ei2"])
    edge, edge_r = U.reverse(ei2)
    assert same(edge, g["edge"]) and same(edge_r, g["edge_r"])
    assert same(U.degree(pos, 3), g["degree"])
    ei_new, x_new, ei2_new = U.sample_block(dev(np.array([0, 1])), 3, pos, ei2)
    assert same(ei_new, g["sb_ei"]) and same(x_new, g["sb_x"]) and same(ei2_new, g["sb_ei2"])
    assert same(U.set_mul(dev(np.array([5, 7])), dev(np.array([1, 2, 3]))), g["set_mul"])
    assert same(U.check_in_set(dev(np.array([1, 2, 3, 2])), dev(np.array([2, 2, 9]))), g["check_in_set"])
    m = U.idx2mask(5, dev(np.array([1, 3])))
    assert m.dtype == torch.bool and same(m, g["idx2mask"])


def test_ragged_golden(U, golden):
    """Irregular inputs: duplicates, self-loop edges, isolated nodes, empty pred / empty pos lists, n_node
    smaller than the largest id."""
    g = golden("ragged.npz")
    k = 0
    while f"c{k}_n" in g.files:
        n = int(g[f"c{k}_n"][0])
        pos, pred = dev(g[f"c{k}_pos"]), dev(g[f"c{k}_pred"])
        ei2 = U.get_ei2(n, pos, pred)
        assert same(ei2, g[f"c{k}_ei2"]), f"case {k} get_ei2"
        if f"c{k}_blocked" in g.files:
            blk = dev(g[f"c{k}_blocked"])
            if f"c{k}_blockei2" in g.files:
                assert same(U.blockei2(ei2, blk), g[f"c{k}_blockei2"]), f"case {k} blockei2 (structured tag)"
                assert same(U.blockei2(ei2.contiguous(), blk), g[f"c{k}_blockei2"]), f"case {k} blockei2 (plain)"
            n_sb = g[f"c{k}_sb_x"].shape[0]
            ei_new, x_new, _ = U.sample_block(blk, n_sb, pos, None)
            assert same(ei_new, g[f"c{k}_sb_ei"]) and same(x_new, g[f"c{k}_sb_x"]), f"case {k} sample_block"
            assert same(U.degree(pos, g[f"c{k}_degree"].shape[0]), g[f"c{k}_degree"]), f"case {k} degree"
        k += 1
    assert k >= 6


def test_fb_pages_food_index_golden(U, fb):
    """configs[0]: the three wedge indices, the train batch's sample_block and reverse, by sha256 of the
    int64 bytes the reference produced."""
    n = int(fb["num_nodes"][0])
    for s in range(3):
        ei, pred, pos1 = fb_split(fb, s)
        ei2 = U.get_ei2(n, dev(ei), dev(pred))
        assert tuple(ei2.shape) == tuple(fb[f"ei2_{s}_shape"])
        assert sha(ei2) == str(fb[f"ei2_{s}_sha"])
    ei, pred, _ = fb_split(fb, 0)
    assert same(U.degree(dev(ei), n), fb["x0"].astype(np.int64))
    ei2 = U.get_ei2(n, dev(ei), dev(pred))
    idx1 = dev(fb["idx1"].astype(np.int64))
    ei_new, x_new, ei2_new = U.sample_block(idx1, n, dev(ei), ei2)
    assert sha(ei_new) == str(fb["sb_ei_sha"]) and same(x_new, fb["sb_x"].astype(np.int64))
    assert sha(ei2_new) == str(fb["sb_ei2_sha"]) and ei2_new.is_contiguous()
    e, er = U.reverse(ei2_new)
    assert sha(e) == str(fb["rev_edge_sha"]) and sha(er) == str(fb["rev_edge_r_sha"])
    # implicit index: same wedge count, same tensor once materialised
    wi = U.blockei2(U.get_ei2_implicit(n, dev(ei), dev(pred)), idx1)
    assert wi.num_wedges() == ei2_new.shape[1]
    assert sha(wi.materialize()) == str(fb["sb_ei2_sha"])


def test_basegraph_preprocess_split_degree_feature_golden(U, fb):
    """SURVEY 8 row a8: the PRODUCT BaseGraph (TwoWL/operators/datasets.py) built from the reference's own split
    (golden edge_pos / edge_neg / num_pos / num_neg), through preprocess() and setPosDegreeFeature(), against what the reference's
    BaseGraph produced from the same inputs (datasets.py:44-114, frozen by oracle/gen_golden.py): pos1s and ei2s by sha256 of
    the int64 bytes, x / ys / max_x / edge_indexs directly, and the split() / dataset() containers."""
    import TwoWL.operators.datasets as D
    n = int(fb["num_nodes"][0])
    ep, en = dev(fb["edge_pos"].astype(np.int64)), dev(fb["edge_neg"].astype(np.int64))
    num_pos, num_neg = torch.from_numpy(fb["num_pos"]), torch.from_numpy(fb["num_neg"])
    for pattern in ("2wl_l", "2wl_l_implicit"):
        bg = D.BaseGraph(torch.zeros((n, 0), device="cuda"), None, ep, en, num_pos, num_neg, pattern)
        assert bg.num_nodes == n and bg.max_x is None
        bg.preprocess()
        bg.setPosDegreeFeature()
        assert bg.max_x == int(fb["max_x"][0])
        for s in range(3):
            ei, pred, pos1 = fb_split(fb, s)
            assert same(bg.edge_indexs[s], ei)
            assert tuple(bg.pos1s[s].shape) == pos1.shape and bg.pos1s[s].dtype == torch.int64
            assert sha(bg.pos1s[s]) == str(fb[f"pos1_{s}_sha"])
            assert same(bg.x[s], fb[f"x{s}"].astype(np.int64)) and bg.x[s].dtype == torch.int64
            assert bg.edge_attrs[s].dtype == torch.float32 and bool((bg.edge_attrs[s] == 1).all())
            assert bg.edge_attrs[s].shape[0] == ei.shape[1]
            ei2 = bg.ei2s[s] if pattern == "2wl_l" else bg.ei2s[s].materialize()
            assert tuple(ei2.shape) == tuple(fb[f"ei2_{s}_shape"]) and sha(ei2) == str(fb[f"ei2_{s}_sha"])
            assert np.array_equal(ei2[:, :64].cpu().numpy(), fb[f"ei2_{s}_head"])
            assert np.array_equal(ei2[:, -64:].cpu().numpy(), fb[f"ei2_{s}_tail"])
        # labels: train = zeros for the negatives only (datasets.py:84), val / test = ones then zeros
        assert bg.ys[0].shape == (int(fb["num_neg"][0]), 1) and not bool(bg.ys[0].any())
        assert bg.ys[1].shape == (int(fb["num_pos"][1] + fb["num_neg"][1]), 1)
        assert bg.ys[2].dtype == torch.float32 and np.array_equal(bg.ys[2].cpu().numpy(), fb["test_y"])
        # containers: split(i) -> dataset(x, na, ei, ea, pos1, y, ei2) exactly as train.py / TwoWL_work.py:40-46 use them
        for s in range(3):
            ds = D.dataset(*bg.split(s))
            assert ds.x is bg.x[s] and ds.na is None and ds.ei is bg.edge_indexs[s] and ds.ea is bg.edge_attrs[s]
            assert ds.pos1 is bg.pos1s[s] and ds.y is bg.ys[s] and ds.ei2 is bg.ei2s[s]
        assert "BaseGraph object" in bg.toString()


# ------------------------------------------------------------------------------ seeded random vs oracle

@pytest.mark.parametrize("n,e,p,seed", [(50, 400, 300, 0), (1000, 6000, 6000, 1), (17, 0, 5, 2), (40, 64, 0, 3),
                                        (5000, 60000, 20000, 4)])
def test_get_ei2_random_vs_oracle(U, n, e, p, seed):
    rng = np.random.default_rng(seed)
    # skewed endpoints (hubs) so that long in/out lists and multi-tile segments occur
    pick = lambda m: np.minimum((rng.pareto(1.2, size=m) * n / 20).astype(np.int64), n - 1)
    pos = np.stack([pick(e), pick(e)])
    pred = np.stack([pick(p), pick(p)])
    ref = O.get_ei2(n, pos, pred)
    got = U.get_ei2(n, dev(pos), dev(pred))
    assert same(got, ref)
    if e:
        blk = rng.choice(e, size=max(1, e // 7), replace=False)
        assert same(U.blockei2(got, dev(blk)), O.blockei2(ref, blk))
        r1, r2 = U.reverse(got)
        o1, o2 = O.reverse(ref)
        assert same(r1, o1) and same(r2, o2)


def test_index_operators_hypothesis_graphs(U):
    """Property test (SURVEY 4 / 7 "hypothesis-generated graphs"): on arbitrary small inputs - empty edge or prediction lists,
    isolated nodes, multi-edges, self loops, blocked ids that repeat - every integer operator equals the oracle bit for bit, on
    the doubled layout (where blockei2 regenerates the join) and on raw, odd-sized lists (where it compacts the tensor)."""
    from hypothesis import given, settings, strategies as st, HealthCheck

    @st.composite
    def graphs(draw):
        n = draw(st.integers(1, 24))
        node = st.integers(0, n - 1)
        und_e = draw(st.lists(st.tuples(node, node), min_size=0, max_size=40))
        und_p = draw(st.lists(st.tuples(node, node), min_size=0, max_size=20))
        doubled = draw(st.booleans())
        seed = draw(st.integers(0, 2 ** 16))
        return n, und_e, und_p, doubled, seed

    @settings(max_examples=60, deadline=None, suppress_health_check=list(HealthCheck))
    @given(graphs())
    def run(case):
        n, und_e, und_p, doubled, seed = case
        rng = np.random.default_rng(seed)
        e = np.array(und_e, dtype=np.int64).reshape(-1, 2).T
        p = np.array(und_p, dtype=np.int64).reshape(-1, 2).T
        pos, pred = (O.double(e), O.double(p)) if doubled else (e, p)
        E = pos.shape[1]
        ref = O.get_ei2(n, pos, pred)
        got = U.get_ei2(n, dev(pos), dev(pred))
        assert same(got, ref)
        assert same(U.degree(dev(pos), n), O.degree(pos, n))
        if E:
            k = int(rng.integers(1, E + 1))
            blk = rng.integers(0, E, size=k)                      # repeats allowed
            assert same(U.blockei2(got, dev(blk)), O.blockei2(ref, blk))
            uniq = np.unique(blk)
            g_ei, g_x, g_ei2 = U.sample_block(dev(uniq), n, dev(pos), got)
            o_ei, o_x, o_ei2 = O.sample_block(uniq, n, pos, ref)
            assert same(g_ei, o_ei) and same(g_x, o_x) and same(g_ei2, o_ei2)
            again = U.blockei2(g_ei2, dev(blk))                   # blocking an already blocked index
            assert same(again, O.blockei2(o_ei2, blk))
        r1, r2 = U.reverse(got)
        o1, o2 = O.reverse(ref)
        assert same(r1, o1) and same(r2, o2)
        if e.shape[1]:
            assert same(U.double(dev(e)), O.double(e))
            ids = rng.integers(0, max(e.shape[1], 1), size=5)
            assert same(U.double(dev(ids), for_index=True), O.double(ids, for_index=True))

    run()


@pytest.mark.parametrize("world", [2, 3, 7])
def test_get_ei2_rank_slices_concatenate_to_the_reference_order(U, world):
    """SURVEY 8(e): every rank fills its own wedge range; the rank-order concatenation is get_ei2 bit for bit."""
    rng = np.random.default_rng(world)
    n = 500
    und = np.concatenate([rng.integers(0, n, size=(2, 2500)), np.stack([np.zeros(300, np.int64), rng.integers(1, n, 300)])], axis=1)
    pos, pred = O.synthetic_split(n, und, seed=world)                 # node 0 is a hub: its segment spans several ranks' ranges
    dpos, dpred = dev(pos), dev(pred)
    full = U.get_ei2(n, dpos, dpred)
    parts = [U.get_ei2_shard(n, dpos, dpred, r, world) for r in range(world)]
    assert all(p[2] == full.shape[1] for p in parts)
    assert [p[1] for p in parts] == [full.shape[1] * r // world for r in range(world)]
    assert torch.equal(torch.cat([p[0] for p in parts], dim=1), full)
    assert np.array_equal(full.cpu().numpy(), O.get_ei2(n, pos, pred))


def test_check_in_set_duplicates_and_degree(U):
    rng = np.random.default_rng(7)
    t = rng.integers(0, 500, size=10000)
    s = rng.integers(0, 600, size=300)   # duplicates count twice (the reference sums the equality matrix)
    assert same(U.check_in_set(dev(t), dev(s)), O.check_in_set(t, s))
    ei = rng.integers(0, 3000, size=(2, 200000))
    assert same(U.degree(dev(ei), 3000), O.degree(ei, 3000))
    assert same(U.degree(dev(ei), 100), np.bincount(ei[1][ei[1] < 100], minlength=100))  # out-of-range dropped


def test_csr_build_is_a_stable_sort(U):
    from twowl_b200 import ops
    rng = np.random.default_rng(11)
    for n, nk in [(1, 1), (2047, 3), (2049, 70000), (300000, 1 << 20), (1000003, 257)]:
        keys = rng.integers(0, nk + 3, size=n)        # some keys out of range: they sort last
        ptr, ids = ops.csr_build(dev(keys), nk)
        kk = np.where(keys < nk, keys, nk)
        ref = np.argsort(kk, kind="stable")
        assert np.array_equal(ids.cpu().numpy(), ref.astype(np.int32)), (n, nk)
        refptr = np.concatenate([[0], np.cumsum(np.bincount(kk[kk < nk], minlength=nk))])
        assert np.array_equal(ptr.cpu().numpy(), refptr), (n, nk)


def test_full_size_properties(U):
    """BASELINE-scale property checks that need no oracle: wedge count identity, sortedness by centre,
    blockei2 == boolean mask, reverse is an involution pair."""
    rng = np.random.default_rng(5)
    n, m = 200000, 1500000
    und = rng.integers(0, n, size=(2, m))
    pos, pred = O.synthetic_split(n, und[:, : m // 2], seed=1)
    # cap T: keep only low-degree nodes' edges out of the way by using the uniform graph (T ~ sum deg^2)
    dpos, dpred = dev(pos), dev(pred)
    ei2 = U.get_ei2(n, dpos, dpred)
    cin = torch.bincount(dpos[1], minlength=n)
    cout = torch.bincount(torch.cat((dpos[0], dpred[0])), minlength=n)
    assert ei2.shape[1] == int((cin * cout).sum())
    centre = dpos[1][ei2[0]]
    assert bool((centre[1:] >= centre[:-1]).all())                       # centre ascending
    src_all = torch.cat((dpos[0], dpred[0]))
    assert bool((src_all[ei2[1]] == centre).all())                       # every wedge is a real join
    blk = dev(rng.choice(pos.shape[1], size=pos.shape[1] // 10, replace=False))
    mask = torch.zeros(pos.shape[1], dtype=torch.bool, device="cuda")
    mask[blk] = True
    assert torch.equal(U.blockei2(ei2, blk), ei2[:, ~mask[ei2[0]]])
    e, er = U.reverse(ei2)
    assert torch.equal(e[0] ^ 1, ei2[0]) and torch.equal(er[1] ^ 1, ei2[1])
    assert torch.equal(e[1], ei2[1]) and torch.equal(er[0], ei2[0])


# ------------------------------------------------------------------------------ floating-point kernels

def _csr_from(rows, cols, M):
    order = np.argsort(rows, kind="stable")
    ptr = np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=M))]).astype(np.int64)
    return dev(ptr), dev(cols[order].astype(np.int32))


@pytest.mark.parametrize("C", [4, 24, 64, 132, 256, 520])
def test_seg_reduce_vs_fp64(U, C):
    from twowl_b200 import ops
    rng = np.random.default_rng(C)
    M, nnz = 3000, 40000
    M += M % 2
    rows = np.minimum((rng.pareto(1.0, size=nnz) * 40).astype(np.int64), M - 1)
    cols = rng.integers(0, M, size=nnz)
    ptr, col = _csr_from(rows, cols, M)
    X = r32(torch.randn(M, C, dtype=torch.float64))       # exactly representable in fp32: no input rounding
    sc = r32(torch.rand(M, dtype=torch.float64) + 0.1)
    bias = r32(torch.randn(C, dtype=torch.float64))
    mask = rng.random(M) < 0.2
    order = np.argsort(rows, kind="stable")
    r_s, c_s = torch.from_numpy(rows[order]), torch.from_numpy(cols[order])
    for flip, row_flip in [(0, 0), (1, 0), (0, 1)]:
        tgt = r_s ^ row_flip
        s = c_s ^ flip
        keep = (s != tgt) & ~torch.from_numpy(mask)[c_s]
        ref = torch.zeros(M, C, dtype=torch.float64).index_add_(0, tgt[keep], sc[s[keep]].unsqueeze(1) * X[s[keep]])
        ref = sc.unsqueeze(1) * ref + (sc ** 2).unsqueeze(1) * X + bias
        # the same sum over the absolute values of its terms, and the longest sum (+ the roundings inside one term): the fp32
        # summation bound of helpers.assert_close - nothing relative to the tensor's largest element
        absum = torch.zeros(M, C, dtype=torch.float64).index_add_(0, tgt[keep], sc[s[keep]].unsqueeze(1) * X[s[keep]].abs())
        absum = sc.unsqueeze(1) * absum + (sc ** 2).unsqueeze(1) * X.abs() + bias.abs()
        nterms = int(torch.bincount(tgt[keep], minlength=M).max()) + 6
        kw = dict(flip=flip, row_flip=row_flip, src_scale=sc.float().cuda(), dst_scale=sc.float().cuda(), skip_self=True,
                  self_mode=1, bias=bias.float().cuda(), skip_mask=dev(mask.astype(np.uint8)))
        got = ops.seg_reduce(ptr, col, M, X.float().cuda(), **kw)
        assert_close(got, ref, absum=absum, nterms=nterms, what=f"seg_reduce C={C} flip={flip} row_flip={row_flip}")
        # with the long-row plan (rows > TWOWL_LONG_ROW entries are cut into chunks): same values, and repeatable
        plan = ops.seg_plan(ptr, M, nnz)
        assert int(plan[0]) >= 1, "the test graph must contain long rows"
        got2 = ops.seg_reduce(ptr, col, M, X.float().cuda(), plan=plan, **kw)
        assert_close(got2, ref, absum=absum, nterms=nterms, what=f"seg_reduce planned C={C}")
        assert torch.equal(got2, ops.seg_reduce(ptr, col, M, X.float().cuda(), plan=ops.seg_plan(ptr, M, nnz), **kw))
        # dinv: exact integer degree
        d = ops.gcn_dinv(ptr, col, M, flip=flip, row_flip=row_flip, skip_mask=dev(mask.astype(np.uint8)))
        deg = torch.bincount(tgt[keep], minlength=M).double() + 1
        assert_close(d, deg.pow(-0.5), rtol=2e-7, atol=0, what="gcn_dinv")


@pytest.mark.parametrize("C", [24, 64, 128, 260])
def test_seg_reduce_dual_output(U, C):
    """One pass over the mated 2-row blocks gives both directions' sums: bit-identical to the two separate passes."""
    from twowl_b200 import ops
    rng = np.random.default_rng(C + 1)
    N, R, nnz = 1500, 4000, 30000
    rows = np.minimum((rng.pareto(1.0, size=nnz) * 30).astype(np.int64), N - 1)
    cols = rng.integers(0, R, size=nnz)
    ptr, col = _csr_from(rows, cols, N)
    X = torch.randn(R, C).cuda()
    s_r, s_f = torch.rand(R).cuda() + 0.1, torch.rand(R).cuda() + 0.1
    mask = dev((rng.random(R) < 0.2).astype(np.uint8))
    for plan in (None, ops.seg_plan(ptr, N, nnz)):
        a = ops.seg_reduce(ptr, col, N, X, plan=plan, flip=0, src_scale=s_r, skip_mask=mask)
        b = ops.seg_reduce(ptr, col, N, X, plan=plan, flip=1, src_scale=s_f, skip_mask=mask)
        a2, b2 = ops.seg_reduce(ptr, col, N, X, plan=plan, src_scale=s_r, skip_mask=mask, dual=True, src_scale2=s_f)
        assert torch.equal(a, a2) and torch.equal(b, b2)
        # the mates' rows from a SECOND matrix (dS_f from dO_f and dS_r from dO_r in one pass over a node's out-list)
        Y = torch.randn(R, C).cuda()
        c = ops.seg_reduce(ptr, col, N, Y, plan=plan, flip=1, src_scale=s_f)
        a3, c3 = ops.seg_reduce(ptr, col, N, X, plan=plan, src_scale=s_r, dual=True, src_scale2=s_f, X_mate=Y)
        assert torch.equal(ops.seg_reduce(ptr, col, N, X, plan=plan, flip=0, src_scale=s_r), a3) and torch.equal(c, c3)


@pytest.mark.parametrize("C", [24, 64])
def test_seg_reduce_row_range_is_the_full_result_on_that_range(U, C):
    """twowl_seg_args.row_begin / row_end (a node block of a row-sharded job): the rows inside the range equal the full launch's
    bit for bit - long rows included - and the rows outside are not touched."""
    from twowl_b200 import ops
    rng = np.random.default_rng(C + 7)
    M, nnz = 3000, 50000
    rows = np.minimum((rng.pareto(1.0, size=nnz) * 40).astype(np.int64), M - 1)
    cols = rng.integers(0, M, size=nnz)
    ptr, col = _csr_from(rows, cols, M)
    X = torch.randn(M, C).cuda()
    sc = (torch.rand(M) + 0.1).cuda()
    bias = torch.randn(C).cuda()
    plan = ops.seg_plan(ptr, M, nnz)
    assert int(plan[0]) >= 1
    kw = dict(plan=plan, src_scale=sc, dst_scale=sc, skip_self=True, self_mode=1, bias=bias)
    full = ops.seg_reduce(ptr, col, M, X, **kw)
    for lo, hi in ((0, 1000), (1000, 2001), (2001, M), (5, 5), (0, M)):
        out = torch.full((M, C), -123.0, device="cuda")
        ops.seg_reduce(ptr, col, M, X, out=out, rows=(lo, hi), **kw)
        assert torch.equal(out[lo:hi], full[lo:hi])
        assert bool((out[:lo] == -123.0).all()) and bool((out[hi:] == -123.0).all())


def test_index_guard_wraps_negative_ids_and_asserts_on_the_rest(U):
    """x[idx] of model.py:78 / utils.py:55: ids in [-num, 0) wrap, anything else outside [0, num) is an IndexError in the
    reference - here a device-side assertion (no host sync on the good path); checked in a subprocess, the assertion poisons the
    CUDA context."""
    import subprocess
    import sys
    from twowl_b200 import ops
    idx = torch.tensor([0, 5, -1, -6, 3], device="cuda")
    assert ops.index_guard(idx, 6).tolist() == [0, 5, 5, 0, 3]
    assert ops.index_guard(idx[::2], 6).tolist() == [0, 5, 3]          # strided view
    import os
    pkg = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "link-prediction-gnn_b200")
    code = ("import sys, torch; sys.path.insert(0, %r); from twowl_b200 import ops; "
            "ops.index_guard(torch.tensor([0, 6], device='cuda'), 6); torch.cuda.synchronize()" % (pkg,))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and ("out of range" in r.stderr or "device-side assert" in r.stderr or "Assertion" in r.stderr), r.stderr[-2000:]
    import TwoWL.model.model  # noqa: F401  (pos out of range -> IndexError once per pair table)
    from twowl_b200 import graph as G
    with pytest.raises(IndexError):
        G.pair_table(torch.tensor([[0, 7], [7, 0]], device="cuda"), 7)


@pytest.mark.parametrize("M,C,p,relu", [(1, 4, 0.0, True), (620, 64, 0.0, False), (6576, 24, 0.0, True),
                                        (100003, 128, 0.0, True), (5000, 32, 0.5, True), (777, 1024, 0.0, True)])
def test_graphnorm_fwd_bwd(U, M, C, p, relu):
    from twowl_b200 import functional as F2
    torch.manual_seed(M + C)
    x = (torch.randn(M, C, dtype=torch.float64) * 2 + 3).requires_grad_(True)
    w = (torch.rand(C, dtype=torch.float64) + 0.5).requires_grad_(True)
    b = torch.randn(C, dtype=torch.float64).requires_grad_(True)
    a = (torch.rand(C, dtype=torch.float64) + 0.5).requires_grad_(True)
    add = torch.randn(M, C, dtype=torch.float64).requires_grad_(True)
    gx, gw, gb, ga, gadd = [t.detach().float().cuda().requires_grad_(True) for t in (x, w, b, a, add)]
    out, _ = F2.graphnorm_act(gx, gw, gb, ga, gadd, 1e-5, p, 1234, relu)
    gout = torch.randn(M, C, dtype=torch.float64)
    out.backward(gout.float().cuda())
    if p == 0.0:
        ref = O.graph_norm(x, w, b, a)
        ref = (torch.relu(ref) if relu else ref) + add
        ref.backward(gout)
        assert_close(out, ref, atol=1e-5, what="graphnorm out")
        scale = lambda t: float(t.abs().max())
        for name, g, r in (("dx", gx, x), ("dw", gw, w), ("db", gb, b), ("dms", ga, a), ("dadd", gadd, add)):
            assert_close(g.grad, r.grad, rtol=1e-5, atol=1e-5 * max(scale(r.grad), 1.0), what="graphnorm " + name)
    else:
        y = O.graph_norm(x, w, b, a).detach()
        o = (out - gadd).detach().cpu().double()
        kept = o != 0
        frac = float(kept.double().mean()) / float((y > 0).double().mean())
        assert abs(frac - (1 - p)) < 0.02, frac                                # keep rate
        assert_close(o[kept], (torch.relu(y) / (1 - p))[kept], atol=1e-5, what="dropout scaling")
        dropped = ~kept & (y > 0.1)                                             # dropped elements pass no gradient
        ref_dx = torch.autograd.grad(O.graph_norm(x, w, b, a), x, gout * kept / (1 - p))[0]
        assert_close(gx.grad, ref_dx, rtol=1e-5, atol=1e-5 * float(ref_dx.abs().max()), what="dropout dx")
        assert int(dropped.sum()) > 0
        # same seed -> same mask; different seed -> different mask
        out2, _ = F2.graphnorm_act(gx, gw, gb, ga, gadd, 1e-5, p, 1234, relu)
        out3, _ = F2.graphnorm_act(gx, gw, gb, ga, gadd, 1e-5, p, 99, relu)
        assert torch.equal(out, out2) and not torch.equal(out, out3)


@pytest.mark.parametrize("M,Ci,Co", [(1, 4, 4), (620, 64, 24), (6576, 24, 24), (4097, 128, 128), (1000, 256, 36),
                                     (50000, 64, 64), (129, 32, 32), (70001, 64, 128), (3000, 128, 64), (257, 96, 48)])
@pytest.mark.parametrize("impl", [0, 2])
def test_linear_fwd_bwd(U, M, Ci, Co, impl, monkeypatch):
    """impl 0 = SIMT FFMA tiles; impl 2 = tcgen05 3xTF32 where the shape is supported (64x64, 128x128->SIMT, ...)."""
    from twowl_b200 import functional as F2
    from twowl_b200 import ops
    monkeypatch.setattr(ops, "LINEAR_IMPL", impl)
    torch.manual_seed(M)
    x = r32(torch.randn(M, Ci, dtype=torch.float64)).requires_grad_(True)
    w = r32(torch.randn(Co, Ci, dtype=torch.float64)).requires_grad_(True)
    g = r32(torch.randn(M, Co, dtype=torch.float64))
    (x @ w.t()).backward(g)
    gx, gw = x.detach().float().cuda().requires_grad_(True), w.detach().float().cuda().requires_grad_(True)
    z = F2.linear(gx, gw)
    z.backward(g.float().cuda())
    # sums of Ci / Co / M products: fp32 summation bound over the absolute terms (+ the split-tf32 product bound on the tensor
    # cores; the weight gradient always runs the SIMT split-K kernel)
    xa, wa, ga = x.detach().abs(), w.detach().abs(), g.abs()
    mma = impl != 0
    assert_close(z, (x @ w.t()).detach(), absum=xa @ wa.t(), nterms=Ci + 2, mma=mma, what="linear fwd")
    assert_close(gx.grad, x.grad, absum=ga @ wa, nterms=Co + 2, mma=mma, what="linear dX")
    assert_close(gw.grad, w.grad, absum=ga.t() @ xa, nterms=M + 2, what="linear dW")


@pytest.mark.parametrize("mated", [False, True])
def test_pair_init_readout_embedding(U, mated):
    from twowl_b200 import functional as F2
    from twowl_b200 import graph as G
    torch.manual_seed(3)
    N, R, C, V, L = 500, 4000, 24, 37, 300
    X = r32(torch.randn(N, C, dtype=torch.float64)).requires_grad_(True)
    pos = torch.randint(0, N, (R, 2))
    if mated:   # the doubled layout of utils.py:81-90: rows 2k / 2k+1 = (u,v) / (v,u) -> one-pass backward
        pos[1::2] = pos[0::2].flip(1)
    idx = torch.randint(0, R, (2 * L,))
    idx[5] = idx[4]
    idx[10] = idx[2]                                   # duplicates: gradients must add up
    w = r32(torch.randn(1, C, dtype=torch.float64)).requires_grad_(True)
    b = r32(torch.randn(1, dtype=torch.float64)).requires_grad_(True)
    emb = r32(torch.randn(V, C, dtype=torch.float64)).requires_grad_(True)
    deg = torch.randint(0, V, (N,))

    def graph(X, w, b, emb):
        h0 = emb[deg] + X
        H = h0[pos[:, 0]] * h0[pos[:, 1]]
        h = H[idx]
        return (h[0::2] * h[1::2]) @ w.t() + b
    ref = graph(X, w, b, emb)
    gout = r32(torch.randn(L, 1, dtype=torch.float64))
    ref.backward(gout)
    # the same graph on the absolute values: every op is a product or a sum with coefficient +1, so its outputs / gradients
    # are the sums of the ABSOLUTE terms of the outputs / gradients above - the `absum` of helpers.assert_close
    leaves = [t.detach().abs().requires_grad_(True) for t in (X, w, b, emb)]
    aref = graph(*leaves)
    aref.backward(gout.abs())
    cnt = torch.bincount(pos.reshape(-1), minlength=N) * int(torch.bincount(idx, minlength=R).max())
    nt = {"dX": int(cnt.max()) + 8, "dw": L + 8, "db": L, "demb": int(torch.bincount(deg, weights=cnt.double(), minlength=V).max()) + 8}

    c = lambda t: t.detach().float().cuda().requires_grad_(True)
    gX, gw, gb, gemb = c(X), c(w), c(b), c(emb)
    pt = G.pair_table(pos.cuda(), N)
    g0 = F2.embedding(gemb, deg.cuda()) + gX
    assert pt.mated == mated
    gH = F2.pair_init(g0, pt.src, pt.dst, pt.ptr_s, pt.ids_s, pt.plan_s, pt.ptr_d, pt.ids_d, pt.plan_d, pt.mated)
    out = F2.readout(gH, idx.cuda(), gw, gb)
    out.backward(gout.float().cuda())
    assert_close(out, ref.detach(), absum=aref.detach(), nterms=C + 8, what="readout fwd")
    for (name, g, r), a in zip((("dX", gX, X), ("dw", gw, w), ("db", gb, b), ("demb", gemb, emb)), leaves):
        assert_close(g.grad, r.grad, absum=a.grad, nterms=nt[name], what=name)


@pytest.mark.parametrize("M,Kd,Nd,nsrc,ngather,stats", [
    (1, 64, 64, 1, 0, False), (127, 32, 32, 1, 1, True), (128, 64, 64, 2, 2, False), (129, 64, 32, 1, 1, True),
    (1000, 32, 64, 2, 1, False), (40001, 64, 64, 1, 1, True), (40001, 64, 64, 2, 2, False), (5000, 64, 128, 1, 2, True),
    (300000, 64, 64, 1, 1, True),
    # widths beyond one K-slab / one column window, and widths that are not multiples of 16 / 32 (fb: channels_2wl = 24)
    (3001, 24, 24, 1, 1, True), (3001, 24, 24, 2, 2, False), (777, 20, 36, 1, 0, True), (20001, 128, 128, 1, 1, True),
    (20001, 128, 128, 2, 2, False), (9001, 256, 256, 1, 1, True), (9001, 256, 256, 2, 2, False), (5000, 96, 48, 2, 1, False),
    (5000, 128, 64, 1, 0, False), (5000, 64, 256, 1, 2, True),
])
def test_pair_conv_tcgen05_vs_fp64(U, M, Kd, Nd, nsrc, ngather, stats):
    """The fused tensor-core kernel (3xTF32 GEMM + row scale + gathered-row epilogue + GraphNorm statistics)."""
    from twowl_b200 import ops
    if not ops.pair_conv_supported(Kd, Nd, nsrc):
        pytest.skip("shape not covered by the tcgen05 kernel")
    torch.manual_seed(M + Kd + Nd)
    NT = 777
    A = [r32(torch.randn(M, Kd, dtype=torch.float64)) for _ in range(nsrc)]
    rs = [r32(torch.rand(M, dtype=torch.float64) * (torch.rand(M) > 0.3)) for _ in range(nsrc)]   # zeros occur (selfw = 0 rows)
    W = [r32(torch.randn(Kd, Nd, dtype=torch.float64) / Kd ** 0.5) for _ in range(nsrc)]          # stored [Kd, Nd]: w_kn = 1
    T = [r32(torch.randn(NT, Nd, dtype=torch.float64)) for _ in range(ngather)]
    idx = [torch.randint(-1, NT, (M,)) for _ in range(ngather)]
    coef = [r32(torch.rand(M, dtype=torch.float64)) for _ in range(ngather)]
    bias = r32(torch.randn(Nd, dtype=torch.float64))
    ref = bias.expand(M, Nd).clone()
    absum = bias.abs().expand(M, Nd).clone()            # the same sum over the absolute values of its terms
    for s in range(nsrc):
        ref += (rs[s].unsqueeze(1) * A[s]) @ W[s]
        absum += (rs[s].unsqueeze(1) * A[s].abs()) @ W[s].abs()
    for g in range(ngather):
        ok = idx[g] >= 0
        ref[ok] += coef[g][ok].unsqueeze(1) * T[g][idx[g][ok]]
        absum[ok] += coef[g][ok].unsqueeze(1) * T[g][idx[g][ok]].abs()
    nterms = nsrc * Kd + ngather + 4
    c = lambda t: t.float().cuda().contiguous()
    for w_kn in (1, 0):
        Wd = [c(w) if w_kn else c(w.t()) for w in W]
        ms = torch.rand(Nd) + 0.5
        args = ([c(a) for a in A], Wd, [w_kn] * nsrc)
        kw = dict(row_scale=[c(r) for r in rs], gathers=[(c(T[g]), idx[g].int().cuda(), c(coef[g])) for g in range(ngather)],
                  bias=c(bias), stats_mean_scale=ms.cuda() if stats else None, eps=1e-5)
        res = ops.pair_conv(*args, **kw)
        out = res[0] if stats else res
        assert_close(out, ref, absum=absum, nterms=nterms, mma=True, what=f"pair_conv out w_kn={w_kn}")
        if stats:
            mean = ref.mean(0)
            var = ((ref - mean * ms.double()) ** 2).mean(0)
            # the column mean inherits the mean of the elements' bounds (its own accumulation runs in double)
            assert_close(res[1][:Nd], mean, absum=absum.mean(0), nterms=nterms, mma=True, what="pair_conv mean")
            # d(inv_std)/inv_std = -d(var) / (2 (var + eps)), |d var| <= 2 mean(|o - a*mean| * bound): first-order propagation of the same bounds
            dev_ = (ref - mean * ms.double()).abs()
            dvar = 2 * (dev_ * absum).mean(0) + 2 * dev_.mean(0) * ms.double() * absum.mean(0)
            inv = (var + 1e-5).rsqrt()
            assert_close(res[1][Nd:], inv, absum=inv * dvar / (2 * (var + 1e-5)), nterms=nterms, mma=True, what="pair_conv inv_std")
            # the raw column moments a row-sharded caller sums over ranks
            _, mom = ops.pair_conv(*args, **kw, want_moments=True)
            assert_close(mom[:Nd], ref.sum(0), absum=absum.sum(0), nterms=nterms, mma=True, what="pair_conv moment sum")
            assert_close(mom[Nd:], (ref ** 2).sum(0), absum=(2 * ref.abs() * absum).sum(0), nterms=nterms, mma=True,
                         what="pair_conv moment sumsq")


@pytest.mark.parametrize("M,C", [(2, 64), (126, 32), (130, 64), (40002, 64), (20002, 128), (3002, 24), (9002, 256)])
def test_pair_conv_pair_sum_out_and_its_consumer_are_bit_identical(U, M, C):
    """twowl_conv_args.pair_sum_out: out[k] = result[2k] + result[2k+1], exactly the full-height result's rows added;
    twowl_seg_args.pair_sum = 2 (seg_reduce(x_pairs=True)) on that tensor = pair_sum = 1 on the full-height one, bit for bit."""
    from twowl_b200 import ops
    if not ops.pair_conv_supported(C, C, 2):
        pytest.skip("shape not covered by the tcgen05 kernel")
    torch.manual_seed(M + C)
    NT = 333
    A = [torch.randn(M, C, device="cuda") for _ in range(2)]
    rs = [torch.rand(M, device="cuda") * (torch.rand(M, device="cuda") > 0.3) for _ in range(2)]
    W = [torch.randn(C, C, device="cuda") / C ** 0.5 for _ in range(2)]
    gathers = [(torch.randn(NT, C, device="cuda"), torch.randint(-1, NT, (M,), device="cuda").int(), torch.rand(M, device="cuda"))
               for _ in range(2)]
    full = ops.pair_conv(A, W, [1, 1], row_scale=rs, gathers=gathers)
    half = ops.pair_conv(A, W, [1, 1], row_scale=rs, gathers=gathers, pair_sum_out=True)
    assert half.shape == (M // 2, C) and torch.equal(half, full[0::2] + full[1::2])
    # the consumer: dx[n] = sum over the rows p with src[p] = n of (g[p] + g[p^1]) * x[dst[p]]
    n = 97
    src = torch.randint(0, n, (M,), device="cuda")
    dst = torch.randint(0, n, (M,), device="cuda").int()
    x = torch.randn(n, C, device="cuda")
    ptr, ids = ops.csr_build(src, n)
    plan = ops.seg_plan(ptr, n, M)
    a = ops.seg_reduce(ptr, ids, n, full, plan=plan, X2=x, mul_idx=dst, pair_sum=True)
    b = ops.seg_reduce(ptr, ids, n, half, plan=plan, X2=x, mul_idx=dst, x_pairs=True)
    assert torch.equal(a, b)


@pytest.mark.parametrize("ratio,M", [(3.0, 40001), (10.0, 40001), (30.0, 300000)])
def test_pair_conv_statistics_with_a_large_mean(U, ratio, M):
    """GraphNorm statistics out of pair_conv's epilogue are raw moments: fp32 (sum, sum of squares) per 32-row block, added in
    double, var = E[x^2] - mean^2 in double (SURVEY 7 hard part 4 warns about this form). The rounding of x^2 is relative to
    mean^2, so the variance loses accuracy as |mean| / std grows: bounded here at the ratios a GCNConv output can plausibly
    reach (bias-dominated columns): inv_std within 1e-5 + ratio^2 * 2^-22 relative. (The op-by-op GraphNorm kernel
    twowl_graphnorm_stats uses shifted sums and has no such dependence.)"""
    from twowl_b200 import ops
    torch.manual_seed(int(ratio) + M)
    Kd = Nd = 64
    A = r32(torch.randn(M, Kd, dtype=torch.float64))
    W = r32(torch.randn(Nd, Kd, dtype=torch.float64) / Kd ** 0.5)         # A W^T has unit variance per column
    bias = r32(torch.full((Nd,), ratio, dtype=torch.float64) * (torch.rand(Nd, dtype=torch.float64) * 0.5 + 0.75))
    ms = torch.ones(Nd)
    ref = A @ W.t() + bias
    c = lambda t: t.float().cuda().contiguous()          # noqa: E731
    out, st = ops.pair_conv([c(A)], [c(W)], [0], bias=c(bias), stats_mean_scale=ms.cuda(), eps=1e-5)
    mean = ref.mean(0)
    inv = (((ref - mean) ** 2).mean(0) + 1e-5).rsqrt()
    assert_close(st[:Nd], mean, rtol=1e-6, atol=1e-6, what="mean")
    rel = ((st[Nd:].double().cpu() - inv) / inv).abs().max()
    assert float(rel) <= 1e-5 + ratio ** 2 * 2.0 ** -22, (float(rel), ratio)


@pytest.mark.parametrize("M,C", [(1, 64), (63, 32), (64, 64), (65, 64), (5000, 32), (70001, 64), (400000, 64), (1, 128), (33, 128),
                                 (70001, 128), (300000, 128)])
def test_pair_dw_tcgen05_vs_fp64(U, M, C):
    """[dW_f; dW_r] = [selfw_f*dO_f | selfw_r*dO_r]^T H with MN-major tcgen05 operands."""
    from twowl_b200 import ops
    torch.manual_seed(M + C)
    dOf, dOr, H = (r32(torch.randn(M, C, dtype=torch.float64)) for _ in range(3))
    rsf = r32(torch.rand(M, dtype=torch.float64) * (torch.rand(M) > 0.3))
    rsr = r32(torch.rand(M, dtype=torch.float64))
    ref_f = (rsf.unsqueeze(1) * dOf).t() @ H
    ref_r = (rsr.unsqueeze(1) * dOr).t() @ H
    c = lambda t: t.float().cuda().contiguous()
    gf, gr = ops.pair_dw(c(dOf), c(dOr), c(rsf), c(rsr), c(H))
    # a sum over M rows (dw_tc.cu): C <= 64: two tiles' 2 x 24 truncating accumulate steps (<= 2u each), then 64 drains in fp32
    # registers, then double; C = 128: 8 tiles x 12 truncating steps, then one fp32 read-add-write per 8 tiles per CTA
    # (+ the roundings of the scaled operand); + the split-tf32 product bound (both operands truncated here: 3 * 2^-20)
    kw = dict(nterms=(168 if C <= 64 else 264 + M // (32 * 148 * 8)), mma=True, mma_bound=3 * 2.0 ** -20)
    assert_close(gf, ref_f, absum=(rsf.unsqueeze(1) * dOf.abs()).t() @ H.abs(), what="pair_dw f", **kw)
    assert_close(gr, ref_r, absum=(rsr.unsqueeze(1) * dOr.abs()).t() @ H.abs(), what="pair_dw r", **kw)
    gf2, gr2 = ops.pair_dw(c(dOf), c(dOr), c(rsf), c(rsr), c(H))
    assert torch.equal(gf, gf2) and torch.equal(gr, gr2)      # deterministic


@pytest.mark.parametrize("M,Co,Ci", [(1, 256, 256), (20001, 256, 256), (5000, 384, 128)])
def test_pair_dw_wide_tiles_vs_fp64(U, M, Co, Ci):
    """Layers wider than 128: the weight gradients tiled into 128-column blocks through pitched TMA tensor maps (twowl_pair_dw_ld)."""
    from twowl_b200 import ops
    torch.manual_seed(M + Co)
    dOf, dOr = (r32(torch.randn(M, Co, dtype=torch.float64)) for _ in range(2))
    H = r32(torch.randn(M, Ci, dtype=torch.float64))
    rsf = r32(torch.rand(M, dtype=torch.float64) * (torch.rand(M) > 0.3))
    rsr = r32(torch.rand(M, dtype=torch.float64))
    c = lambda t: t.float().cuda().contiguous()          # noqa: E731
    assert ops.pair_dw_wide_supported(Co, Ci)
    gf, gr = ops.pair_dw_wide(c(dOf), c(dOr), c(rsf), c(rsr), c(H))
    ref_f, ref_r = (rsf.unsqueeze(1) * dOf).t() @ H, (rsr.unsqueeze(1) * dOr).t() @ H
    kw = dict(nterms=264 + M // (32 * 148 * 8), mma=True, mma_bound=3 * 2.0 ** -20)      # the 128-column launches, as test_pair_dw_tcgen05_vs_fp64
    assert_close(gf, ref_f, absum=(rsf.unsqueeze(1) * dOf.abs()).t() @ H.abs(), what="pair_dw_wide f", **kw)
    assert_close(gr, ref_r, absum=(rsr.unsqueeze(1) * dOr.abs()).t() @ H.abs(), what="pair_dw_wide r", **kw)


@pytest.mark.parametrize("M,C,L,p", [(64, 64, 10, 0.0), (5000, 32, 700, 0.3), (70001, 64, 9000, 0.0), (70001, 64, 9000, 0.5),
                                     (40001, 128, 5000, 0.0), (40001, 128, 5000, 0.4)])
def test_pair_dw_gn_matches_two_pass(U, M, C, L, p):
    """twowl_gn2_readout_bwd_rows + _finish + twowl_pair_dw_gn (GraphNorm backward made inside the weight-gradient kernel) against
    the two-pass path twowl_gn2_readout_bwd + twowl_pair_dw: same dO_f, dO_r, dW_f, dW_r and parameter gradients."""
    from twowl_b200 import ops
    torch.manual_seed(M + C + L)
    dev = "cuda"
    Of, Or, H = (torch.randn(M, C, device=dev) for _ in range(3))
    rsf = torch.rand(M, device=dev) * (torch.rand(M, device=dev) > 0.3)
    rsr = torch.rand(M, device=dev)
    pf = tuple(torch.rand(C, device=dev) + 0.5 for _ in range(3))
    pr = tuple(torch.rand(C, device=dev) + 0.5 for _ in range(3))
    sf, sr = ops.graphnorm_stats(Of, pf[2], 1e-5), ops.graphnorm_stats(Or, pr[2], 1e-5)
    idx = torch.randint(0, M, (2 * L,), device=dev)
    idx[3] = idx[1]
    idx[7] = idx[1]                       # a row selected three times: positions add in ascending order
    w = torch.randn(1, C, device=dev)
    dpred = torch.randn(L, device=dev)
    seeds = (1234567, 7654321)
    dxf, dxr, dpf, dpr, dw, db = ops.gn2_readout_bwd(Of, Or, sf, sr, pf, pr, p, seeds[0], seeds[1], True, idx, w, dpred)
    dWf, dWr = ops.pair_dw(dxf, dxr, rsf, rsr, H)
    G, head, nxt, consts, dpf2, dpr2, dw2, db2 = ops.gn2_readout_bwd_prepare(Of, Or, sf, sr, pf, pr, p, seeds[0], seeds[1], True, idx, w,
                                                                           dpred)
    dOf, dOr, dWf2, dWr2 = ops.pair_dw_gn(Of, Or, consts, G, head, nxt, p, seeds[0], seeds[1], True, rsf, rsr, H)
    for a, b in ((dpf, dpf2), (dpr, dpr2), (dw, dw2), (db, db2)):
        assert torch.equal(a, b)
    tol = 1e-5 * max(float(dxf.abs().max()), float(dxr.abs().max()))
    assert_close(dOf, dxf.double().cpu(), rtol=1e-5, atol=tol, what="dO_f on the fly")
    assert_close(dOr, dxr.double().cpu(), rtol=1e-5, atol=tol, what="dO_r on the fly")
    wt = 1e-5 * max(float(dWf.abs().max()), float(dWr.abs().max()), 1.0)
    assert_close(dWf2, dWf.double().cpu(), rtol=1e-5, atol=wt, what="dW_f")
    assert_close(dWr2, dWr.double().cpu(), rtol=1e-5, atol=wt, what="dW_r")
