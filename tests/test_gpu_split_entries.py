"""The pair-level entry points that one GPU and one rank of a row-sharded step share, checked on one GPU against their whole-table
calls: the per-row wedge constants over two ranges of pair rows, the entry-masked gcn_norm degrees over a node range, and the two
pair-layer GraphNorm backwards with the rows cut into two blocks and an all_reduce hook that adds the other block's column sums."""
import numpy as np
import pytest
import torch

from helpers import assert_close

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from twowl_b200 import ops as ops_mod
    return ops_mod


def _doubled(rng, n, k):
    """[2, 2k] int64 with columns 2i = (u, v), 2i+1 = (v, u); node 0 is a hub."""
    u = np.where(rng.random(k) < 0.1, 0, rng.integers(0, n, k))
    v = rng.integers(0, n, k)
    return torch.from_numpy(np.stack([np.stack([u, v], 1).reshape(-1), np.stack([v, u], 1).reshape(-1)])).cuda()


@pytest.mark.parametrize("with_blocked", [False, True])
def test_wedge_prepare_ranges_are_rows_of_the_whole_table(ops, with_blocked):
    from twowl_b200 import graph as G
    from twowl_b200.rowshard import blocks_of
    rng = np.random.default_rng(5 + with_blocked)
    N = 3000
    ws = G.build_wedge_struct(N, _doubled(rng, N, 20000), _doubled(rng, N, 15000))
    E, R = ws.E, ws.R
    blocked = torch.from_numpy((rng.random(E) < 0.3).astype(np.uint8)).cuda() if with_blocked else None
    args = (ws.src, ws.dst_e, E, R, N, blocked, ws.in_ptr)
    full = ops.wedge_prepare(*args)
    assert all(t.shape == (2, R) for t in full[1:])
    cases = [((0, R), (R, R)), ((0, 0), (E, R)), ((0, E), (E, E)), ((2, E - 4), (E + 6, R - 2))]
    cases += [blocks_of(E, R, rank, 3) for rank in range(3)]
    for ranges in cases:
        (lo0, hi0), (lo1, hi1) = ranges
        got = ops.wedge_prepare(*args, ranges=ranges)
        rows = torch.cat((torch.arange(lo0, hi0), torch.arange(lo1, hi1))).cuda()
        assert torch.equal(got[0][:N], full[0][:N]), ranges
        for a, b in zip(got[1:], full[1:]):
            assert torch.equal(a, b[:, rows]), ranges
    for bad in (((1, 4), (R, R)), ((0, E), (0, R)), ((0, R + 2), (R + 2, R + 2))):
        with pytest.raises(RuntimeError, match="even-bounded, ordered"):
            ops.wedge_prepare(*args, ranges=bad)


def test_gcn_dinv_entries_over_a_row_range(ops):
    rng = np.random.default_rng(11)
    N, nnz = 2000, 40000
    rows = np.where(rng.random(nnz) < 0.08, 7, rng.integers(0, N, nnz))   # row 7 is a hub: many 8 x 32-entry iterations
    cols = np.where(rng.random(nnz) < 0.05, rows, rng.integers(0, N, nnz))   # some self loops, which do not count
    order = np.argsort(rows, kind="stable")
    rows, cols = rows[order], cols[order]
    mask = (rng.random(nnz) < 0.25).astype(np.uint8)
    ptr = torch.from_numpy(np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=N))]).astype(np.int64)).cuda()
    col = torch.from_numpy(cols.astype(np.int32)).cuda()
    emask = torch.from_numpy(mask).cuda()
    full = ops.gcn_dinv_entries(ptr, col, N, emask)
    keep = (mask == 0) & (cols != rows)
    deg = torch.from_numpy(np.bincount(rows[keep], minlength=N).astype(np.float64) + 1)
    assert_close(full, deg.pow(-0.5), rtol=2e-7, atol=0, what="gcn_dinv_entries")
    for lo, hi in ((0, N), (17, 1234), (7, 8), (5, 5), (1999, 2000)):
        out = torch.full((N + 5,), -1.0, device="cuda")
        assert ops.gcn_dinv_entries(ptr, col, N, emask, rows=(lo, hi), out=out) is out
        assert torch.equal(out[lo:hi], full[lo:hi])
        assert bool((out[:lo] == -1).all()) and bool((out[hi:] == -1).all())


def _two_block_hook(call, cut, M):
    """call(lo, hi, all_reduce) on the row blocks [0, cut) and [cut, M): a first pass records each block's column sums, a second
    pass adds the other block's sums in the hook - the all-reduce of two ranks. -> the two blocks' results."""
    own = [None, None]
    blocks = ((0, cut), (cut, M))

    def record(b):
        def hook(t):
            own[b] = t.clone()
        return hook

    for b, (lo, hi) in enumerate(blocks):
        call(lo, hi, record(b))
    return [call(lo, hi, lambda t, b=b: t.add_(own[1 - b])) for b, (lo, hi) in enumerate(blocks)]


def _close(got, ref, what):
    tol = 1e-5 * max(float(ref.abs().max()), 1e-30)
    assert_close(got, ref.double().cpu(), rtol=1e-5, atol=tol, what=what)


@pytest.mark.parametrize("M,C,cut", [(64, 32, 20), (40000, 64, 14000), (30001, 128, 15000)])
def test_graphnorm_bwd2_two_blocks_match_the_whole_table(ops, M, C, cut):
    torch.manual_seed(M + C)
    dev = "cuda"
    Of, Or, g = (torch.randn(M, C, device=dev) for _ in range(3))
    pf = tuple(torch.rand(C, device=dev) + 0.5 for _ in range(3))
    pr = tuple(torch.rand(C, device=dev) + 0.5 for _ in range(3))
    sf, sr = ops.graphnorm_stats(Of, pf[2], 1e-5), ops.graphnorm_stats(Or, pr[2], 1e-5)
    # no dropout: a block's dropout mask is keyed by its own row ids, so only p = 0 makes the blocks a cut of the whole table
    full = ops.graphnorm_bwd2(Of, Or, g, sf, sr, pf, pr, 0.0, 1, 2, True)
    a, b = _two_block_hook(lambda lo, hi, ar: ops.graphnorm_bwd2(Of[lo:hi], Or[lo:hi], g[lo:hi], sf, sr, pf, pr, 0.0, 1, 2, True, M, ar),
                           cut, M)
    for i, what in ((0, "dxf"), (1, "dxr")):
        _close(torch.cat((a[i], b[i])), full[i], what)
    for i, what in ((2, "dparams_f"), (3, "dparams_r")):
        assert torch.equal(a[i], b[i])             # both blocks finish from the same summed sums
        _close(a[i], full[i], what)


@pytest.mark.parametrize("M,C,L,cut", [(64, 32, 10, 20), (40000, 64, 5000, 14000), (30001, 128, 4000, 15000)])
def test_gn2_readout_bwd_prepare_two_blocks_match_the_whole_table(ops, M, C, L, cut):
    torch.manual_seed(M + C + L)
    dev = "cuda"
    Of, Or = (torch.randn(M, C, device=dev) for _ in range(2))
    pf = tuple(torch.rand(C, device=dev) + 0.5 for _ in range(3))
    pr = tuple(torch.rand(C, device=dev) + 0.5 for _ in range(3))
    sf, sr = ops.graphnorm_stats(Of, pf[2], 1e-5), ops.graphnorm_stats(Or, pr[2], 1e-5)
    # both rows of a link in one block (as a row-sharded step cuts the table), some rows selected several times
    in_a = torch.rand(L, device=dev) < cut / M
    in_a[:3], in_a[3] = True, False
    base = torch.where(in_a, 0, cut).unsqueeze(1)
    n = torch.where(in_a, cut, M - cut).unsqueeze(1)
    idx = (base + (torch.rand(L, 2, device=dev) * n).long()).reshape(-1)
    idx[1] = idx[0]
    idx[4] = idx[0]
    w = torch.randn(1, C, device=dev)
    dpred = torch.randn(L, device=dev)
    full = ops.gn2_readout_bwd_prepare(Of, Or, sf, sr, pf, pr, 0.0, 1, 2, True, idx, w, dpred)

    def block(lo, hi, ar):
        own = ((idx >= lo) & (idx < hi)).reshape(L, 2).all(1).repeat_interleave(2)
        idx_l = torch.where(own, idx - lo, -1)     # a negative id masks the other block's links
        return ops.gn2_readout_bwd_prepare(Of[lo:hi], Or[lo:hi], sf, sr, pf, pr, 0.0, 1, 2, True, idx_l, w, dpred, M, ar), own

    (a, own_a), (b, own_b) = _two_block_hook(block, cut, M)
    assert bool((own_a ^ own_b).all())
    for got, own in ((a, own_a), (b, own_b)):
        assert torch.equal(got[0][own], full[0][own])          # G: per position, no reduction
    for i, what in ((3, "consts"), (4, "dparams_f"), (5, "dparams_r"), (6, "dw"), (7, "db")):
        assert torch.equal(a[i], b[i])
        _close(a[i], full[i], what)
