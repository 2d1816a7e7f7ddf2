"""The depth-1 pair layer's H at half height (twowl::pair_init_layer_readout): on a mated pair table rows 2k and 2k+1 of
H = x[src] * x[dst] are the same bits, so every consumer reads ONE row per pair. Each half-height kernel is checked bit for bit
against the full-height kernel on the expanded H = Hh.repeat_interleave(2, 0)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from twowl_b200 import ops as ops_mod
    return ops_mod


def _mated(n, pairs, gen):
    """A mated table: rows 2k / 2k+1 are (u,v) / (v,u)."""
    u = torch.randint(0, n, (pairs,), generator=gen)
    v = torch.randint(0, n, (pairs,), generator=gen)
    src = torch.stack([u, v], 1).reshape(-1).int().cuda()
    dst = torch.stack([v, u], 1).reshape(-1).int().cuda()
    return src, dst


@pytest.mark.parametrize("C", [4, 64, 128, 260])
def test_pair_init_half_is_both_rows_of_the_full(ops, C):
    gen = torch.Generator().manual_seed(C)
    src, dst = _mated(977, 5003, gen)
    x = torch.randn(977, C, generator=gen).cuda()
    full = ops.pair_init_fwd(x, src, dst)
    half = ops.pair_init_fwd(x, src, dst, pairs=True)
    assert half.shape == (full.shape[0] // 2, C)
    assert torch.equal(half, full[0::2]) and torch.equal(half, full[1::2])


@pytest.mark.parametrize("C", [24, 64, 128, 260])
def test_seg_reduce_dual_over_one_row_per_pair(ops, C):
    """twowl_seg_args.pair_sum = 2 with the dual output: both outputs as from the full-height 2-row blocks, with and without the
    long-row plan and with a blocked-entry mask."""
    rng = np.random.default_rng(C + 7)
    N, P, nnz = 1500, 2000, 30000
    R = 2 * P
    rows = np.minimum((rng.pareto(1.0, size=nnz) * 30).astype(np.int64), N - 1)
    cols = rng.integers(0, R, size=nnz)
    order = np.argsort(rows, kind="stable")
    ptr = torch.from_numpy(np.concatenate([[0], np.cumsum(np.bincount(rows, minlength=N))]).astype(np.int64)).cuda()
    col = torch.from_numpy(cols[order].astype(np.int32)).cuda()
    Hh = torch.randn(P, C).cuda()
    H = Hh.repeat_interleave(2, 0)
    s_r, s_f = torch.rand(R).cuda() + 0.1, torch.rand(R).cuda() + 0.1
    for plan in (None, ops.seg_plan(ptr, N, nnz)):
        for mask in (None, torch.from_numpy((rng.random(R) < 0.2).astype(np.uint8)).cuda()):
            a, b = ops.seg_reduce(ptr, col, N, H, plan=plan, src_scale=s_r, skip_mask=mask, dual=True, src_scale2=s_f)
            a2, b2 = ops.seg_reduce(ptr, col, N, Hh, plan=plan, src_scale=s_r, skip_mask=mask, dual=True, src_scale2=s_f,
                                    x_pairs=True)
            assert torch.equal(a, a2) and torch.equal(b, b2)


@pytest.mark.parametrize("P,C", [(1, 64), (63, 32), (4099, 32), (20001, 64), (20033, 128), (150001, 64)])
def test_pair_conv_forward_with_a_at_half_height(ops, P, C):
    """twowl_conv_args.a_pairs: out and the GraphNorm statistics as with A = Hh.repeat_interleave(2, 0). P (= M/2) is not a
    multiple of 64, so the last tile is partial; C = 128 runs two column windows."""
    M = 2 * P
    torch.manual_seed(P + C)
    NT = 777
    Hh = torch.randn(P, C, device="cuda")
    H = Hh.repeat_interleave(2, 0)
    rs = torch.rand(M, device="cuda") * (torch.rand(M, device="cuda") > 0.3)
    W = torch.randn(C, C, device="cuda") / C ** 0.5
    bias = torch.randn(C, device="cuda")
    gm = torch.rand(C, device="cuda") + 0.5
    g = (torch.randn(NT, C, device="cuda"), torch.randint(-1, NT, (M,), device="cuda").int(), torch.rand(M, device="cuda"))
    O, st = ops.pair_conv([H], [W], [0], row_scale=[rs], gathers=[g], bias=bias, stats_mean_scale=gm, eps=1e-5)
    O2, st2 = ops.pair_conv([Hh], [W], [0], row_scale=[rs], gathers=[g], bias=bias, stats_mean_scale=gm, eps=1e-5, a_pairs=True)
    assert O2.shape == (M, C)
    assert torch.equal(O, O2) and torch.equal(st, st2)


@pytest.mark.parametrize("P,C,L,p", [(32, 64, 10, 0.0), (2500, 32, 700, 0.3), (35001, 64, 9000, 0.5), (20001, 128, 5000, 0.4)])
@pytest.mark.parametrize("inplace", [False, True])
def test_pair_dw_gn_with_h_at_half_height(ops, P, C, L, p, inplace):
    """twowl_pair_dw_gn with h_pairs = 1: dO_f, dO_r, dW_f, dW_r as with H = Hh.repeat_interleave(2, 0)."""
    M = 2 * P
    torch.manual_seed(M + C + L)
    dev = "cuda"
    Of, Or = (torch.randn(M, C, device=dev) for _ in range(2))
    Hh = torch.randn(P, C, device=dev)
    H = Hh.repeat_interleave(2, 0)
    rsf = torch.rand(M, device=dev) * (torch.rand(M, device=dev) > 0.3)
    rsr = torch.rand(M, device=dev)
    pf = tuple(torch.rand(C, device=dev) + 0.5 for _ in range(3))
    pr = tuple(torch.rand(C, device=dev) + 0.5 for _ in range(3))
    sf, sr = ops.graphnorm_stats(Of, pf[2], 1e-5), ops.graphnorm_stats(Or, pr[2], 1e-5)
    idx = torch.randint(0, M, (2 * L,), device=dev)
    w = torch.randn(1, C, device=dev)
    dpred = torch.randn(L, device=dev)
    seeds = (1234567, 7654321)
    G, head, nxt, consts, *_ = ops.gn2_readout_bwd_prepare(Of, Or, sf, sr, pf, pr, p, seeds[0], seeds[1], True, idx, w, dpred)
    ref = ops.pair_dw_gn(Of, Or, consts, G, head, nxt, p, seeds[0], seeds[1], True, rsf, rsr, H)
    Of2, Or2 = (Of.clone(), Or.clone()) if inplace else (Of, Or)
    got = ops.pair_dw_gn(Of2, Or2, consts, G, head, nxt, p, seeds[0], seeds[1], True, rsf, rsr, Hh, inplace=inplace)
    for a, b in zip(ref, got):
        assert torch.equal(a, b)
    if inplace:
        assert got[0].data_ptr() == Of2.data_ptr() and got[1].data_ptr() == Or2.data_ptr()
