"""The differentiable TwoWL ops, registered as torch custom ops (namespace ``twowl::``) whose
forward AND backward are calls into libtwowl_b200.so. They replace, on the hot path, the
torch_geometric / torch_scatter kernels the reference reaches through
TwoWL/model/model.py:37-38,53-55,73,75,77-83.

Every backward is the hand-derived transpose of its forward over the same index (CSR by source
instead of CSR by target), not an autograd trace of torch ops.
"""
from __future__ import annotations

from typing import List, Optional, Tuple

import torch
from torch import Tensor

from . import ops

# ------------------------------------------------------------------------------ linear (GCNConv.lin)


@torch.library.custom_op("twowl::linear", mutates_args=())
def linear(x: Tensor, weight: Tensor) -> Tensor:
    """PyG Linear(bias=False): x @ weight.T, fp32-exact accumulation."""
    return ops.linear_fwd(x.contiguous(), weight.contiguous())


@linear.register_fake
def _(x, weight):
    return x.new_empty((x.shape[0], weight.shape[0]))


def _linear_setup(ctx, inputs, output):
    ctx.save_for_backward(*inputs)


def _linear_bwd(ctx, g):
    x, w = ctx.saved_tensors
    g = g.contiguous()
    dx = ops.linear_bwd_input(g, w.contiguous()) if ctx.needs_input_grad[0] else None
    dw = ops.linear_bwd_weight(g, x.contiguous()) if ctx.needs_input_grad[1] else None
    return dx, dw


linear.register_autograd(_linear_bwd, setup_context=_linear_setup)

# ------------------------------------------------------------------------------ explicit GCN propagate


@torch.library.custom_op("twowl::gcn_aggregate", mutates_args=())
def gcn_aggregate(z: Tensor, bias: Tensor, dinv: Tensor, ptr: Tensor, col: Tensor, plan: Optional[Tensor], tptr: Tensor,
                  tcol: Tensor, tplan: Optional[Tensor], mask: Optional[Tensor], flip: int, row_flip: int,
                  emask: Optional[Tensor] = None, temask: Optional[Tensor] = None) -> Tensor:
    """out[m] = dinv[m] * sum_{k in row m^row_flip, s=col[k]^flip != m, !mask[col[k]]} dinv[s] z[s]
               + dinv[m]^2 z[m] + bias   (PyG GCNConv.propagate with gcn_norm, SURVEY.md 3.4)."""
    return ops.seg_reduce(ptr, col, z.shape[0], z.contiguous(), plan=plan, flip=flip, row_flip=row_flip, src_scale=dinv,
                          dst_scale=dinv, skip_self=True, self_mode=1, bias=bias, skip_mask=mask, entry_mask=emask)


@gcn_aggregate.register_fake
def _(z, bias, dinv, ptr, col, plan, tptr, tcol, tplan, mask, flip, row_flip, emask=None, temask=None):
    return torch.empty_like(z)


def _gcn_setup(ctx, inputs, output):
    z, bias, dinv, ptr, col, plan, tptr, tcol, tplan, mask, flip, row_flip, emask, temask = inputs
    ctx.save_for_backward(dinv, tptr, tcol, tplan, mask, temask)
    ctx.flip, ctx.row_flip = flip, row_flip


def _gcn_bwd(ctx, g):
    dinv, tptr, tcol, tplan, mask, temask = ctx.saved_tensors
    g = g.contiguous()
    dz = dbias = None
    if ctx.needs_input_grad[0]:
        # transpose: rows by SOURCE; the roles of flip / row_flip swap; the column mask becomes a row mask
        dz = ops.seg_reduce(tptr, tcol, g.shape[0], g, plan=tplan, flip=ctx.row_flip, row_flip=ctx.flip, src_scale=dinv,
                            dst_scale=dinv, skip_self=True, self_mode=1, row_skip_mask=mask, entry_mask=temask)
    if ctx.needs_input_grad[1]:
        dbias = ops.colsum(g)
    return (dz, dbias) + (None,) * 12


gcn_aggregate.register_autograd(_gcn_bwd, setup_context=_gcn_setup)

# ------------------------------------------------------------------------------ structured pair-level propagate


@torch.library.custom_op("twowl::wedge_aggregate", mutates_args=())
def wedge_aggregate(z: Tensor, bias: Tensor, in_ptr: Tensor, in_ids: Tensor, in_plan: Optional[Tensor], out_ptr: Tensor,
                    out_ids: Tensor, out_plan: Optional[Tensor], centre: Tensor, dinv: Tensor, selfw: Tensor, dst_e: Tensor, blocked: Optional[Tensor], n_edge: int,
                    n_node: int, direction: int) -> Tensor:
    """Pair-level GCNConv for a wedge index that is the full join of get_ei2 minus blocked source edges:
    S[i] = sum over unblocked in-edges of i; out[b] = dinv[b] S[centre[b]] + selfw[b] z[b] + bias
    (DESIGN.md 'Factorised pair aggregation'). direction 0 = edge2, 1 = edge2_r of utils.py:71-78."""
    z = z.contiguous()
    S = ops.seg_reduce(in_ptr, in_ids, n_node, z, plan=in_plan, flip=1 - direction, src_scale=dinv, skip_mask=blocked)
    return ops.wedge_apply_fwd(S, z, centre, dinv, selfw, bias)


@wedge_aggregate.register_fake
def _(z, bias, in_ptr, in_ids, in_plan, out_ptr, out_ids, out_plan, centre, dinv, selfw, dst_e, blocked, n_edge, n_node,
      direction):
    return torch.empty_like(z)


def _wedge_setup(ctx, inputs, output):
    (z, bias, in_ptr, in_ids, in_plan, out_ptr, out_ids, out_plan, centre, dinv, selfw, dst_e, blocked, n_edge, n_node,
     direction) = inputs
    ctx.save_for_backward(out_ptr, out_ids, out_plan, dinv, selfw, dst_e, blocked)
    ctx.meta = (n_edge, n_node, direction)


def _wedge_bwd(ctx, g):
    out_ptr, out_ids, out_plan, dinv, selfw, dst_e, blocked = ctx.saved_tensors
    n_edge, n_node, direction = ctx.meta
    g = g.contiguous()
    dz = dbias = None
    if ctx.needs_input_grad[0]:
        dS = ops.seg_reduce(out_ptr, out_ids, n_node, g, plan=out_plan, flip=direction, src_scale=dinv)
        dz = ops.wedge_apply_bwd(dS, g, dst_e, blocked, n_edge, n_node, dinv, selfw, direction)
    if ctx.needs_input_grad[1]:
        dbias = ops.colsum(g)
    return (dz, dbias) + (None,) * 14


wedge_aggregate.register_autograd(_wedge_bwd, setup_context=_wedge_setup)

# ------------------------------------------------------------------------------ GraphNorm + Dropout + ReLU


@torch.library.custom_op("twowl::graphnorm_act", mutates_args=())
def graphnorm_act(x: Tensor, weight: Tensor, bias: Tensor, mean_scale: Tensor, addend: Optional[Tensor], eps: float,
                  p_drop: float, seed: int, relu: bool) -> Tuple[Tensor, Tensor]:
    """relu?(dropout_p(GraphNorm(x))) + addend?  ->  (out, stats[2C] = (mean, inv_std))."""
    x = x.contiguous()
    stats = ops.graphnorm_stats(x, mean_scale, eps)
    out = ops.graphnorm_apply(x, stats, weight, bias, mean_scale, p_drop, seed, relu,
                              None if addend is None else addend.contiguous())
    return out, stats


@graphnorm_act.register_fake
def _(x, weight, bias, mean_scale, addend, eps, p_drop, seed, relu):
    return torch.empty_like(x), x.new_empty((2 * x.shape[1],))


def _gn_setup(ctx, inputs, output):
    x, weight, bias, mean_scale, addend, eps, p_drop, seed, relu = inputs
    ctx.save_for_backward(x, weight, bias, mean_scale, output[1])
    ctx.meta = (p_drop, seed, relu)
    ctx.has_addend = addend is not None
    ctx.mark_non_differentiable(output[1])
    ctx.set_materialize_grads(False)


def _gn_bwd(ctx, g, _g_stats):
    x, weight, bias, mean_scale, stats = ctx.saved_tensors
    p_drop, seed, relu = ctx.meta
    g = g.contiguous()
    dx, dparams = ops.graphnorm_bwd(x.contiguous(), g, stats, weight, bias, mean_scale, p_drop, seed, relu)
    C = x.shape[1]
    return (dx, dparams[:C], dparams[C:2 * C], dparams[2 * C:3 * C], g if ctx.has_addend else None, None, None, None, None)


graphnorm_act.register_autograd(_gn_bwd, setup_context=_gn_setup)

# ------------------------------------------------------------------------------ node-attribute input (model.py:47-51,71)

_K_CHUNK = 1024   # widest reduction dimension one linear launch takes


def _chunks(F: int):
    return [(k, min(k + _K_CHUNK, F)) for k in range(0, F, _K_CHUNK)]


def _pad4(t: Tensor) -> Tensor:
    """[rows, F] -> contiguous [rows, F rounded up to a multiple of 4] (zero columns: they add nothing to a product)."""
    F = t.shape[1]
    if F % 4 == 0:
        return t.contiguous()
    out = t.new_zeros((t.shape[0], F + (4 - F % 4)))
    out[:, :F] = t
    return out


@torch.library.custom_op("twowl::node_feat_input", mutates_args=())
def node_feat_input(node_feat: Tensor, weight: Tensor, bias: Tensor, eps: float, p_in: float, seed_in: int, p_out: float,
                    seed_out: int) -> Tuple[Tensor, Tensor, Tensor]:
    """Dropout(p_out)(LayerNorm(Linear(Dropout(p_in)(node_feat)))) of model.py:47-51 -> (x [N, c], z = the Linear's product before
    the bias [N, c], stats [N, 2]); any feature width F (padded to a multiple of 4, cut into <= 1024-column slabs)."""
    xin = _pad4(node_feat if p_in == 0.0 else ops.dropout(node_feat, p_in, seed_in))
    w = _pad4(weight)
    z = None
    for lo, hi in _chunks(xin.shape[1]):
        part = ops.linear_fwd(xin[:, lo:hi].contiguous(), w[:, lo:hi].contiguous())
        z = part if z is None else z.add_(part)
    y, stats = ops.bias_layernorm_fwd(z, bias.contiguous(), eps, p_out, seed_out)
    return y, z, stats


@node_feat_input.register_fake
def _(node_feat, weight, bias, eps, p_in, seed_in, p_out, seed_out):
    y = node_feat.new_empty((node_feat.shape[0], weight.shape[0]))
    return y, torch.empty_like(y), node_feat.new_empty((node_feat.shape[0], 2))


def _nf_setup(ctx, inputs, output):
    node_feat, weight, bias, eps, p_in, seed_in, p_out, seed_out = inputs
    ctx.save_for_backward(node_feat, bias, output[1], output[2])
    ctx.meta = (weight.shape[1], p_in, seed_in, p_out, seed_out)
    ctx.mark_non_differentiable(output[1], output[2])
    ctx.set_materialize_grads(False)


def _nf_bwd(ctx, g, *_unused):
    node_feat, bias, z, stats = ctx.saved_tensors
    F, p_in, seed_in, p_out, seed_out = ctx.meta
    dz = ops.bias_layernorm_bwd(g.contiguous(), z, bias.contiguous(), stats, p_out, seed_out)
    dbias = ops.colsum(dz)
    xin = _pad4(node_feat if p_in == 0.0 else ops.dropout(node_feat, p_in, seed_in))      # the mask is regenerated from its seed
    dW = torch.cat([ops.linear_bwd_weight(dz, xin[:, lo:hi].contiguous()) for lo, hi in _chunks(xin.shape[1])], dim=1)[:, :F]
    return None, dW.contiguous(), dbias, None, None, None, None, None


node_feat_input.register_autograd(_nf_bwd, setup_context=_nf_setup)

# ------------------------------------------------------------------------------ embedding lookup


@torch.library.custom_op("twowl::embedding", mutates_args=())
def embedding(weight: Tensor, x: Tensor) -> Tensor:
    return ops.gather_rows(weight.contiguous(), x)


@embedding.register_fake
def _(weight, x):
    return weight.new_empty((x.numel(), weight.shape[1]))


def _emb_setup(ctx, inputs, output):
    ctx.save_for_backward(inputs[1])
    ctx.rows = inputs[0].shape[0]


def _emb_bwd(ctx, g):
    (x,) = ctx.saved_tensors
    ptr, ids = ops.csr_build(x.reshape(-1), ctx.rows)   # rows = degree values: extremely skewed, so plan it
    plan = ops.seg_plan(ptr, ctx.rows, ids.numel())
    return ops.seg_reduce(ptr, ids, ctx.rows, g.contiguous(), plan=plan), None


embedding.register_autograd(_emb_bwd, setup_context=_emb_setup)

# ------------------------------------------------------------------------------ pair init


@torch.library.custom_op("twowl::pair_init", mutates_args=())
def pair_init(x: Tensor, src: Tensor, dst: Tensor, ptr_s: Tensor, ids_s: Tensor, plan_s: Optional[Tensor], ptr_d: Tensor,
              ids_d: Tensor, plan_d: Optional[Tensor], mated: bool = False) -> Tensor:
    """H[p] = x[src[p]] * x[dst[p]] (model.py:75); (ptr_s, ids_s) / (ptr_d, ids_d) = pair rows grouped by
    src / dst node, used by the backward. mated: rows 2k / 2k+1 are (u,v) / (v,u) (utils.py:81-90)."""
    return ops.pair_init_fwd(x.contiguous(), src, dst)


@pair_init.register_fake
def _(x, src, dst, ptr_s, ids_s, plan_s, ptr_d, ids_d, plan_d, mated=False):
    return x.new_empty((src.numel(), x.shape[1]))


def _pi_setup(ctx, inputs, output):
    ctx.save_for_backward(*inputs[:9])
    ctx.mated = bool(inputs[9])


def _pi_bwd(ctx, g):
    x, src, dst, ptr_s, ids_s, plan_s, ptr_d, ids_d, plan_d = ctx.saved_tensors
    g = g.contiguous()
    N = x.shape[0]
    # dx[n] = sum_{p: src[p]=n} g[p]*x[dst[p]] + sum_{p: dst[p]=n} g[p]*x[src[p]]
    if ctx.mated:
        # the pairs with dst = n are the mates p^1 of the pairs with src = n, and src[p^1] = dst[p]:
        # dx[n] = sum_{p: src[p]=n} (g[p] + g[p^1]) * x[dst[p]] - one pass, g read once as 2-row blocks
        dx = ops.seg_reduce(ptr_s, ids_s, N, g, plan=plan_s, X2=x, mul_idx=dst, pair_sum=True)
    else:
        dx = ops.seg_reduce(ptr_s, ids_s, N, g, plan=plan_s, X2=x, mul_idx=dst)
        ops.seg_reduce(ptr_d, ids_d, N, g, plan=plan_d, X2=x, mul_idx=src, out=dx, accumulate=True)
    return (dx,) + (None,) * 9


pair_init.register_autograd(_pi_bwd, setup_context=_pi_setup)


def batch_pair_init(x: Tensor, pairs: Tensor) -> Tensor:
    """pair_init for a batch of query pairs (int64 [B, 2]): x[pairs[:, 0]] * x[pairs[:, 1]]. The by-source / by-destination CSRs the
    backward reads are built here for this batch, not cached: they live as long as the batch."""
    N, B = x.shape[0], pairs.shape[0]
    ptr_s, ids_s = ops.csr_build(pairs[:, 0], N)
    ptr_d, ids_d = ops.csr_build(pairs[:, 1], N)
    return pair_init(x, ops.narrow_i32(pairs[:, 0]), ops.narrow_i32(pairs[:, 1]), ptr_s, ids_s, ops.seg_plan(ptr_s, N, B), ptr_d, ids_d,
                     ops.seg_plan(ptr_d, N, B), False)

# ------------------------------------------------------------------------------ common-neighbour sum (TwoWL/model/ncn.py)


@torch.library.custom_op("twowl::cn_aggregate", mutates_args=())
def _cn_aggregate(h: Tensor, cn_ptr: Tensor, cn_ids: Tensor, cn_pair: Tensor, plan: Tensor) -> Tensor:
    return ops.seg_reduce(cn_ptr, cn_ids, cn_ptr.numel() - 1, h.contiguous(), plan=plan)


@_cn_aggregate.register_fake
def _(h, cn_ptr, cn_ids, cn_pair, plan):
    return h.new_empty((cn_ptr.shape[0] - 1, h.shape[1]))


def _cna_setup(ctx, inputs, output):
    h, cn_ptr, cn_ids, cn_pair, plan = inputs
    ctx.save_for_backward(cn_ids, cn_pair)
    ctx.N = h.shape[0]


def _cna_bwd(ctx, g):
    cn_ids, cn_pair = ctx.saved_tensors
    N = ctx.N
    # dh[w] = sum of g[p] over the pairs p whose list holds w: the entries grouped by node with a stable sort, so that each node's
    # pairs come in ascending order, then one segmented sum
    tptr, tids = ops.csr_build(cn_ids.to(torch.int64), N)
    tcol = ops.gather_cols(tids, cn_pair.to(torch.int64))
    return ops.seg_reduce(tptr, tcol, N, g.contiguous(), plan=ops.seg_plan(tptr, N, tcol.numel())), None, None, None, None


_cn_aggregate.register_autograd(_cna_bwd, setup_context=_cna_setup)


def cn_aggregate(h: Tensor, cn) -> Tensor:
    """out [P, C] with out[p] = sum of h[w] over w in CN(p), for cn an ops.CommonNeighbors of P pairs and h [N, C] (C % 4 == 0).
    Forward and backward are segmented sums in a fixed order (no float atomics): bitwise repeatable."""
    P = cn.num_pairs
    return _cn_aggregate(h, cn.ptr, cn.ids, cn.pair, ops.seg_plan(cn.ptr, P, cn.ids.numel()))

# ------------------------------------------------------------------------------ readout


@torch.library.custom_op("twowl::readout", mutates_args=())
def readout(h: Tensor, idx: Tensor, weight: Tensor, bias: Tensor) -> Tensor:
    """pred[l] = (h[idx[2l]] * h[idx[2l+1]]) @ weight.T + bias  (model.py:78-83)."""
    return ops.readout_fwd(h.contiguous(), idx, weight.contiguous(), bias)


@readout.register_fake
def _(h, idx, weight, bias):
    return h.new_empty((idx.numel() // 2, 1))


def _ro_setup(ctx, inputs, output):
    ctx.save_for_backward(*inputs)


def _ro_bwd(ctx, g):
    h, idx, weight, bias = ctx.saved_tensors
    dH, dw, db = ops.readout_bwd(h.contiguous(), idx, weight.contiguous(), g.reshape(-1))
    return dH, None, dw, db


readout.register_autograd(_ro_bwd, setup_context=_ro_setup)


# ------------------------------------------------------------------------------ fused structured pair layer
#
# One custom op for  x <- relu(drop(GN_f(conv_f(x, edge2)))) + relu(drop(GN_r(conv_r(x, edge2_r))))  (model.py:77)
# on the structured wedge path: per direction d
#   SH_d = per-node sum of dinv_d * H over the unblocked in-edges          (seg_reduce, N rows)
#   O_d  = selfw_d * (H W_d^T) + dinv_d * (SH_d W_d^T)[centre_d] + bias_d   (tcgen05 GEMM, fused epilogue + GN statistics)
# and the two GraphNorm(+Dropout+ReLU) applications summed. The backward is hand-written from the same pieces.


def _pair_convs_fwd(h, pf, pr, SHf, SHr, centre, dinv, selfw, eps, h_pairs=False):
    """O_d = selfw_d * (h W_d^T) + dinv_d * (SH_d W_d^T)[centre_d] + bias_d and its GraphNorm statistics, both directions:
    -> [(O_f, stats_f, SH_f), (O_r, stats_r, SH_r)]. h_pairs: h holds one row per pair (row r of O uses h[r >> 1])."""
    (wf, bf, gmf), (wr, br, gmr) = pf, pr
    Sf, Sr = ops.linear_fwd(SHf, wf), ops.linear_fwd(SHr, wr)
    outs = []
    for d, (w, b, gm, S, SH) in enumerate(((wf, bf, gmf, Sf, SHf), (wr, br, gmr, Sr, SHr))):
        O, st = ops.pair_conv([h], [w], [0], row_scale=[selfw[d]], gathers=[(S, centre[d], dinv[d])], bias=b,
                              stats_mean_scale=gm, eps=eps, a_pairs=h_pairs)
        outs.append((O, st, SH))
    return outs


@torch.library.custom_op("twowl::pair_layer", mutates_args=())
def pair_layer(h: Tensor, wf: Tensor, bf: Tensor, gwf: Tensor, gbf: Tensor, gmf: Tensor, wr: Tensor, br: Tensor, gwr: Tensor,
               gbr: Tensor, gmr: Tensor, in_ptr: Tensor, in_ids: Tensor, in_plan: Tensor, out_ptr: Tensor, out_ids: Tensor,
               out_plan: Tensor, centre: Tensor, dinv: Tensor, selfw: Tensor, bnode: Tensor, blocked: Optional[Tensor],
               n_node: int, eps: float, p_drop: float, seed_f: int, seed_r: int
               ) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """-> (h_next, O_f, O_r, stats_f, stats_r, SH_f, SH_r); only h_next is differentiable, the rest is saved state."""
    h = h.contiguous()
    # both directions' in-list sums from one pass over the mated 2-row blocks of h: SH_r gathers h[a], SH_f h[a^1]
    SHr, SHf = ops.seg_reduce(in_ptr, in_ids, n_node, h, plan=in_plan, src_scale=dinv[1], skip_mask=blocked, dual=True,
                              src_scale2=dinv[0])
    outs = _pair_convs_fwd(h, (wf, bf, gmf), (wr, br, gmr), SHf, SHr, centre, dinv, selfw, eps)
    hn = ops.graphnorm_apply2(outs[0][0], outs[1][0], outs[0][1], outs[1][1], (gwf, gbf, gmf), (gwr, gbr, gmr), p_drop, seed_f,
                              seed_r, True)
    return hn, outs[0][0], outs[1][0], outs[0][1], outs[1][1], outs[0][2], outs[1][2]


@pair_layer.register_fake
def _(h, wf, bf, gwf, gbf, gmf, wr, br, gwr, gbr, gmr, in_ptr, in_ids, in_plan, out_ptr, out_ids, out_plan, centre, dinv,
      selfw, bnode, blocked, n_node, eps, p_drop, seed_f, seed_r):
    C = wf.shape[0]
    o = h.new_empty((h.shape[0], C))
    return (o, torch.empty_like(o), torch.empty_like(o), h.new_empty((2 * C,)), h.new_empty((2 * C,)),
            h.new_empty((n_node, h.shape[1])), h.new_empty((n_node, h.shape[1])))


def _pl_setup(ctx, inputs, output):
    (h, wf, bf, gwf, gbf, gmf, wr, br, gwr, gbr, gmr, in_ptr, in_ids, in_plan, out_ptr, out_ids, out_plan, centre, dinv,
     selfw, bnode, blocked, n_node, eps, p_drop, seed_f, seed_r) = inputs
    hn, Of, Or, sf, sr, SHf, SHr = output
    ctx.save_for_backward(h, wf, bf, gwf, gbf, gmf, wr, br, gwr, gbr, gmr, out_ptr, out_ids, out_plan, dinv, selfw, bnode,
                          Of, Or, sf, sr, SHf, SHr)
    ctx.meta = (n_node, p_drop, seed_f, seed_r)
    ctx.mark_non_differentiable(Of, Or, sf, sr, SHf, SHr)
    ctx.set_materialize_grads(False)   # no zero-filled [R,C] gradients for the saved-state outputs


def _pl_bwd_core(h, wf, wr, out_ptr, out_ids, out_plan, dinv, selfw, bnode, SHf, SHr, n_node, dOs, dpars, dWs=None, dh_out=None,
                 pair_sum_out=False):
    """Backward of the structured pair-level GCNConv pair from the gradients dO_f, dO_r of its two outputs:
    -> dh and, per direction, (dW, dbias, d gn.weight, d gn.bias, d gn.mean_scale).
    dWs: the (selfw_d * dO_d)^T H parts when the caller already has them (pair_dw_gn)."""
    C = wf.shape[0]
    # both directions' gradient sums from ONE pass over every node's out-list: entry b contributes dinv_f[b] * dO_f[b] to dS_f and
    # dinv_r[b^1] * dO_r[b^1] to dS_r (bit-identical to the two passes with flip = 0 / 1)
    dSs = list(ops.seg_reduce(out_ptr, out_ids, n_node, dOs[0].contiguous(), plan=out_plan, src_scale=dinv[0], dual=True,
                              src_scale2=dinv[1], X_mate=dOs[1].contiguous()))
    # dW_d = (selfw_d * dO_d)^T H + dS_d^T SH_d ;  the gathered part of dH goes through (dS_d W_d)
    if dWs is not None:
        pass
    elif ops.pair_dw_supported(C) and h.shape[1] == C:
        dWs = list(ops.pair_dw(dOs[0], dOs[1], selfw[0], selfw[1], h))
    elif ops.pair_dw_wide_supported(C, h.shape[1]):
        dWs = list(ops.pair_dw_wide(dOs[0].contiguous(), dOs[1].contiguous(), selfw[0], selfw[1], h))
    else:
        dWs = [ops.linear_bwd_weight(dOs[d], h, row_scale=selfw[d]) for d in range(2)]
    res, dSWs = [], []
    for d, (w, SH) in enumerate(((wf, SHf), (wr, SHr))):
        dW = dWs[d] + ops.linear_bwd_weight(dSs[d], SH)
        dSWs.append(ops.linear_bwd_input(dSs[d], w))
        dpar = dpars[d]
        res.append((dW, dpar[3 * C:], dpar[:C], dpar[C:2 * C], dpar[2 * C:3 * C]))
    # pair_sum_out: dh is [R/2, C] and holds dH[2k] + dH[2k+1] - all the pair-init backward wants of it (pair_init_layer_readout)
    dh = ops.pair_conv(dOs, [wf, wr], [1, 1], row_scale=[selfw[0], selfw[1]],
                       gathers=[(dSWs[0], bnode[0], dinv[0]), (dSWs[1], bnode[1], dinv[1])], out=dh_out, pair_sum_out=pair_sum_out)
    return dh, res


def _pl_bwd(ctx, g, *_unused):
    (h, wf, bf, gwf, gbf, gmf, wr, br, gwr, gbr, gmr, out_ptr, out_ids, out_plan, dinv, selfw, bnode, Of, Or, sf, sr, SHf,
     SHr) = ctx.saved_tensors
    n_node, p_drop, seed_f, seed_r = ctx.meta
    g = g.contiguous()
    dOf, dOr, dpf, dpr = ops.graphnorm_bwd2(Of, Or, g, sf, sr, (gwf, gbf, gmf), (gwr, gbr, gmr), p_drop, seed_f, seed_r, True)
    dh, res = _pl_bwd_core(h, wf, wr, out_ptr, out_ids, out_plan, dinv, selfw, bnode, SHf, SHr, n_node, [dOf, dOr], [dpf, dpr])
    return (dh,) + res[0] + res[1] + (None,) * 16


pair_layer.register_autograd(_pl_bwd, setup_context=_pl_setup)


# ------------------------------------------------------------------------------ last pair layer + readout
#
# The LAST conv2s / conv2s_r layer only feeds x[idx] (model.py:77-83): the GraphNorm(+Dropout+ReLU) branches are evaluated
# at the 2L selected rows, h_next [R,C] is never materialised, and the backward starts from a row-sparse gradient.


@torch.library.custom_op("twowl::pair_layer_readout", mutates_args=())
def pair_layer_readout(h: Tensor, wf: Tensor, bf: Tensor, gwf: Tensor, gbf: Tensor, gmf: Tensor, wr: Tensor, br: Tensor, gwr: Tensor,
                       gbr: Tensor, gmr: Tensor, idx: Tensor, pw: Tensor, pb: Tensor, in_ptr: Tensor, in_ids: Tensor,
                       in_plan: Tensor, out_ptr: Tensor, out_ids: Tensor, out_plan: Tensor, centre: Tensor, dinv: Tensor,
                       selfw: Tensor, bnode: Tensor, blocked: Optional[Tensor], n_node: int, eps: float, p_drop: float,
                       seed_f: int, seed_r: int) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """-> (pred [L,1], O_f, O_r, stats_f, stats_r, SH_f, SH_r); only pred is differentiable, the rest is saved state."""
    return _plr_forward(h.contiguous(), wf, bf, gwf, gbf, gmf, wr, br, gwr, gbr, gmr, idx, pw, pb, in_ptr, in_ids, in_plan, centre, dinv,
                        selfw, blocked, n_node, eps, p_drop, seed_f, seed_r)


def _plr_forward(h, wf, bf, gwf, gbf, gmf, wr, br, gwr, gbr, gmr, idx, pw, pb, in_ptr, in_ids, in_plan, centre, dinv, selfw, blocked,
                 n_node, eps, p_drop, seed_f, seed_r, h_pairs=False):
    """h_pairs: h is [R/2, C], one row per pair, standing for rows 2k and 2k+1 of the mated pair table (pair_init_layer_readout)."""
    # both directions' in-list sums from one pass over the mated 2-row blocks of h: SH_r gathers h[a], SH_f h[a^1] (h_pairs: the
    # one row h[a >> 1] feeds both)
    SHr, SHf = ops.seg_reduce(in_ptr, in_ids, n_node, h, plan=in_plan, src_scale=dinv[1], skip_mask=blocked, dual=True,
                              src_scale2=dinv[0], x_pairs=h_pairs)
    outs = _pair_convs_fwd(h, (wf, bf, gmf), (wr, br, gmr), SHf, SHr, centre, dinv, selfw, eps, h_pairs)
    pred = ops.gn2_readout_fwd(outs[0][0], outs[1][0], outs[0][1], outs[1][1], (gwf, gbf, gmf), (gwr, gbr, gmr), p_drop, seed_f,
                               seed_r, True, idx, pw.contiguous(), pb)
    return pred, outs[0][0], outs[1][0], outs[0][1], outs[1][1], outs[0][2], outs[1][2]


@pair_layer_readout.register_fake
def _(h, wf, bf, gwf, gbf, gmf, wr, br, gwr, gbr, gmr, idx, pw, pb, in_ptr, in_ids, in_plan, out_ptr, out_ids, out_plan, centre,
      dinv, selfw, bnode, blocked, n_node, eps, p_drop, seed_f, seed_r):
    C = wf.shape[0]
    o = h.new_empty((h.shape[0], C))
    return (h.new_empty((idx.numel() // 2, 1)), o, torch.empty_like(o), h.new_empty((2 * C,)), h.new_empty((2 * C,)),
            h.new_empty((n_node, h.shape[1])), h.new_empty((n_node, h.shape[1])))


def _plr_setup(ctx, inputs, output):
    (h, wf, bf, gwf, gbf, gmf, wr, br, gwr, gbr, gmr, idx, pw, pb, in_ptr, in_ids, in_plan, out_ptr, out_ids, out_plan, centre,
     dinv, selfw, bnode, blocked, n_node, eps, p_drop, seed_f, seed_r) = inputs
    pred, Of, Or, sf, sr, SHf, SHr = output
    ctx.save_for_backward(h, wf, bf, gwf, gbf, gmf, wr, br, gwr, gbr, gmr, idx, pw, out_ptr, out_ids, out_plan, dinv, selfw,
                          bnode, Of, Or, sf, sr, SHf, SHr)
    ctx.meta = (n_node, p_drop, seed_f, seed_r)
    ctx.mark_non_differentiable(Of, Or, sf, sr, SHf, SHr)
    ctx.set_materialize_grads(False)   # no zero-filled [R,C] gradients for the saved-state outputs


def _plr_bwd(ctx, g, *_unused):
    n_node, p_drop, seed_f, seed_r = ctx.meta
    dh, res, dpw, dpb = _plr_backward(g, ctx.saved_tensors, n_node, p_drop, seed_f, seed_r)
    return (dh,) + res[0] + res[1] + (None, dpw, dpb) + (None,) * 16


def _plr_backward(g, saved, n_node, p_drop, seed_f, seed_r, pair_sum_out=False):
    """Backward of the fused last pair layer + readout from d pred: -> (dh, per-direction parameter gradients, d pred.weight,
    d pred.bias). pair_sum_out: dh is [R/2, C], the sum of the two directions' rows of every pair. h may hold one row per pair
    ([R/2, C], pair_init_layer_readout): only pair_dw_gn reads it then."""
    (h, wf, bf, gwf, gbf, gmf, wr, br, gwr, gbr, gmr, idx, pw, out_ptr, out_ids, out_plan, dinv, selfw, bnode, Of, Or, sf, sr,
     SHf, SHr) = saved
    C = wf.shape[0]
    h_pairs = h.shape[0] != Of.shape[0]
    if h_pairs or (ops.pair_dw_supported(C) and h.shape[1] == C):
        # the dense GraphNorm-backward pass rides on the weight-gradient kernel's shared-memory pass (twowl_pair_dw_gn)
        G, head, nxt, consts, dpf, dpr, dpw, dpb = ops.gn2_readout_bwd_prepare(Of, Or, sf, sr, (gwf, gbf, gmf), (gwr, gbr, gmr),
                                                                               p_drop, seed_f, seed_r, True, idx, pw.contiguous(),
                                                                               g.reshape(-1))
        inplace = ops.INPLACE_BACKWARD and wf.shape[0] == wf.shape[1]
        dOf, dOr, dWf, dWr = ops.pair_dw_gn(Of, Or, consts, G, head, nxt, p_drop, seed_f, seed_r, True, selfw[0], selfw[1], h,
                                            inplace=inplace)
        dWs = [dWf, dWr]
    else:
        inplace = False
        dOf, dOr, dpf, dpr, dpw, dpb = ops.gn2_readout_bwd(Of, Or, sf, sr, (gwf, gbf, gmf), (gwr, gbr, gmr), p_drop, seed_f, seed_r,
                                                           True, idx, pw.contiguous(), g.reshape(-1))
        dWs = None
    dh_out = None
    if inplace:      # h is not read by that launch: dH (or its pair sums, in the first half of the buffer) may take its place
        dh_out = h.view(-1)[:(h.shape[0] // 2) * h.shape[1]].view(h.shape[0] // 2, h.shape[1]) if pair_sum_out and not h_pairs else h
    dh, res = _pl_bwd_core(h, wf, wr, out_ptr, out_ids, out_plan, dinv, selfw, bnode, SHf, SHr, n_node, [dOf, dOr], [dpf, dpr],
                           dWs=dWs, dh_out=dh_out, pair_sum_out=pair_sum_out)
    return dh, res, dpw.reshape(pw.shape), dpb


pair_layer_readout.register_autograd(_plr_bwd, setup_context=_plr_setup)


# The same with the pair init (model.py:75) inside the op, for a model whose ONLY pair layer is that last one (depth2 = 1): then
# the gradient of H = x[src] * x[dst] is consumed by nothing but the pair-init backward, which adds the two directions' rows of
# every pair before anything else - so the input-gradient GEMM writes ONE row per pair (twowl_conv_args.pair_sum_out: half its
# output bytes) and the pair-init backward reads that (twowl_seg_args.pair_sum = 2: half of both of its passes). Same terms, same
# order: bit-identical to pair_init -> pair_layer_readout.


@torch.library.custom_op("twowl::pair_init_layer_readout", mutates_args=())
def pair_init_layer_readout(x: Tensor, src: Tensor, dst: Tensor, ptr_s: Tensor, ids_s: Tensor, plan_s: Optional[Tensor], wf: Tensor,
                            bf: Tensor, gwf: Tensor, gbf: Tensor, gmf: Tensor, wr: Tensor, br: Tensor, gwr: Tensor, gbr: Tensor,
                            gmr: Tensor, idx: Tensor, pw: Tensor, pb: Tensor, in_ptr: Tensor, in_ids: Tensor, in_plan: Tensor,
                            out_ptr: Tensor, out_ids: Tensor, out_plan: Tensor, centre: Tensor, dinv: Tensor, selfw: Tensor,
                            bnode: Tensor, blocked: Optional[Tensor], n_node: int, eps: float, p_drop: float, seed_f: int,
                            seed_r: int) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """-> (pred [L,1], H, O_f, O_r, stats_f, stats_r, SH_f, SH_r); only pred is differentiable, the rest is saved state.
    H is private to the op, and on the mated table its rows 2k and 2k+1 are the same bits: where the weight-gradient kernel
    covers the width it is kept at half height, ONE row per pair ([R/2, C]), and every consumer reads that row for both."""
    h_pairs = _plr_h_pairs(x.shape[1], wf.shape[0])
    h = ops.pair_init_fwd(x.contiguous(), src, dst, pairs=h_pairs)
    return (h,) + _plr_forward(h, wf, bf, gwf, gbf, gmf, wr, br, gwr, gbr, gmr, idx, pw, pb, in_ptr, in_ids, in_plan, centre, dinv,
                               selfw, blocked, n_node, eps, p_drop, seed_f, seed_r, h_pairs)


def _plr_h_pairs(Cin: int, C: int) -> bool:
    """Whether pair_init_layer_readout keeps H at half height: the widths pair_dw_gn covers (other widths compute the weight
    gradient from a full-height H)."""
    return Cin == C and ops.pair_dw_supported(C)


@pair_init_layer_readout.register_fake
def _(x, src, dst, ptr_s, ids_s, plan_s, wf, bf, gwf, gbf, gmf, wr, br, gwr, gbr, gmr, idx, pw, pb, in_ptr, in_ids, in_plan, out_ptr,
      out_ids, out_plan, centre, dinv, selfw, bnode, blocked, n_node, eps, p_drop, seed_f, seed_r):
    C = wf.shape[0]
    h = x.new_empty((src.numel() // 2 if _plr_h_pairs(x.shape[1], C) else src.numel(), x.shape[1]))
    o = x.new_empty((src.numel(), C))
    return (h, x.new_empty((idx.numel() // 2, 1)), o, torch.empty_like(o), x.new_empty((2 * C,)), x.new_empty((2 * C,)),
            x.new_empty((n_node, x.shape[1])), x.new_empty((n_node, x.shape[1])))


def _pilr_setup(ctx, inputs, output):
    (x, src, dst, ptr_s, ids_s, plan_s, wf, bf, gwf, gbf, gmf, wr, br, gwr, gbr, gmr, idx, pw, pb, in_ptr, in_ids, in_plan, out_ptr,
     out_ids, out_plan, centre, dinv, selfw, bnode, blocked, n_node, eps, p_drop, seed_f, seed_r) = inputs
    h, pred, Of, Or, sf, sr, SHf, SHr = output
    ctx.save_for_backward(x, dst, ptr_s, ids_s, plan_s, h, wf, bf, gwf, gbf, gmf, wr, br, gwr, gbr, gmr, idx, pw, out_ptr, out_ids,
                          out_plan, dinv, selfw, bnode, Of, Or, sf, sr, SHf, SHr)
    ctx.meta = (n_node, p_drop, seed_f, seed_r)
    ctx.mark_non_differentiable(h, Of, Or, sf, sr, SHf, SHr)
    ctx.set_materialize_grads(False)


def _pilr_bwd(ctx, _g_h, g, *_unused):
    x, dst, ptr_s, ids_s, plan_s, *saved = ctx.saved_tensors
    n_node, p_drop, seed_f, seed_r = ctx.meta
    dh2, res, dpw, dpb = _plr_backward(g, saved, n_node, p_drop, seed_f, seed_r, pair_sum_out=True)
    # dx[n] = sum over the pair rows p with src[p] = n of (dH[p] + dH[p^1]) * x[dst[p]], the sum read from dh2[p >> 1]
    dx = ops.seg_reduce(ptr_s, ids_s, x.shape[0], dh2, plan=plan_s, X2=x, mul_idx=dst, x_pairs=True)
    return (dx,) + (None,) * 5 + res[0] + res[1] + (None, dpw, dpb) + (None,) * 16


pair_init_layer_readout.register_autograd(_pilr_bwd, setup_context=_pilr_setup)


def pair_layer_supported(wedges, C: int, seq_f, seq_r) -> bool:
    """Structured wedges, equal in/out width, a width the tensor-core kernel covers, ReLU blocks (model.py:62-65)."""
    from .graph import WedgeStruct
    if not isinstance(wedges, WedgeStruct):
        return False
    convf = seq_f.modlist[0]
    if convf.in_channels != C or convf.out_channels != C or seq_r.modlist[0].out_channels != C:
        return False
    if not (isinstance(seq_f.modlist[3], torch.nn.ReLU) and isinstance(seq_r.modlist[3], torch.nn.ReLU)):
        return False
    return ops.pair_conv_supported(C, C, 2) and ops.LINEAR_IMPL != 0


def pair_layer_apply(x, wedges, seq_f, seq_r, training: bool):
    cf, gf, dpf = seq_f.modlist[0], seq_f.modlist[1], seq_f.modlist[2]
    cr, gr = seq_r.modlist[0], seq_r.modlist[1]
    p = dpf.p if (training and dpf.p > 0.0) else 0.0
    seeds = [ops.next_seed() for _ in range(2)] if p > 0.0 else [0, 0]
    _, centre, dinv, selfw, bnode = wedges.prepared()
    out = pair_layer(x, cf.lin.weight, cf.bias, gf.weight, gf.bias, gf.mean_scale, cr.lin.weight, cr.bias, gr.weight, gr.bias,
                     gr.mean_scale, wedges.in_ptr, wedges.in_ids, wedges.in_plan, wedges.out_ptr, wedges.out_ids,
                     wedges.out_plan, centre, dinv, selfw, bnode, wedges.blocked, wedges.n_node, gf.eps, p, seeds[0], seeds[1])
    return out[0]


def pair_layer_readout_apply(x, wedges, seq_f, seq_r, training: bool, idx, pred):
    """Last pair layer fused with the readout: pred(x'[idx] even*odd) of model.py:77-83 without materialising x'."""
    cf, gf, dpf = seq_f.modlist[0], seq_f.modlist[1], seq_f.modlist[2]
    cr, gr = seq_r.modlist[0], seq_r.modlist[1]
    p = dpf.p if (training and dpf.p > 0.0) else 0.0
    seeds = [ops.next_seed() for _ in range(2)] if p > 0.0 else [0, 0]
    _, centre, dinv, selfw, bnode = wedges.prepared()
    out = pair_layer_readout(x, cf.lin.weight, cf.bias, gf.weight, gf.bias, gf.mean_scale, cr.lin.weight, cr.bias, gr.weight,
                             gr.bias, gr.mean_scale, idx, pred.weight, pred.bias, wedges.in_ptr, wedges.in_ids, wedges.in_plan,
                             wedges.out_ptr, wedges.out_ids, wedges.out_plan, centre, dinv, selfw, bnode, wedges.blocked,
                             wedges.n_node, gf.eps, p, seeds[0], seeds[1])
    return out[0]


def pair_init_layer_readout_apply(x, pt, wedges, seq_f, seq_r, training: bool, idx, pred):
    """model.py:75-83 for depth2 = 1 in one op: pair init + the only pair layer + readout (pt: graph.PairTable, doubled layout)."""
    cf, gf, dpf = seq_f.modlist[0], seq_f.modlist[1], seq_f.modlist[2]
    cr, gr = seq_r.modlist[0], seq_r.modlist[1]
    p = dpf.p if (training and dpf.p > 0.0) else 0.0
    seeds = [ops.next_seed() for _ in range(2)] if p > 0.0 else [0, 0]
    _, centre, dinv, selfw, bnode = wedges.prepared()
    out = pair_init_layer_readout(x, pt.src, pt.dst, pt.ptr_s, pt.ids_s, pt.plan_s, cf.lin.weight, cf.bias, gf.weight, gf.bias,
                                  gf.mean_scale, cr.lin.weight, cr.bias, gr.weight, gr.bias, gr.mean_scale, idx, pred.weight,
                                  pred.bias, wedges.in_ptr, wedges.in_ids, wedges.in_plan, wedges.out_ptr, wedges.out_ids,
                                  wedges.out_plan, centre, dinv, selfw, bnode, wedges.blocked, wedges.n_node, gf.eps, p, seeds[0],
                                  seeds[1])
    return out[1]


# ------------------------------------------------------------------------------ loss (train.py:37)


@torch.library.custom_op("twowl::bce_with_logits", mutates_args=())
def _bce_with_logits(logits: Tensor, labels: Tensor) -> Tuple[Tensor, Tensor]:
    loss, dx, _ = ops.bce_logits(logits, labels, want_grad=True)
    return loss.reshape(()), dx


@_bce_with_logits.register_fake
def _(logits, labels):
    return logits.new_empty(()), torch.empty_like(logits)


def _bce_setup(ctx, inputs, output):
    ctx.save_for_backward(output[1])
    ctx.mark_non_differentiable(output[1])
    ctx.set_materialize_grads(False)


def _bce_bwd(ctx, g, _g_dx):
    (dx,) = ctx.saved_tensors
    return dx * g, None


_bce_with_logits.register_autograd(_bce_bwd, setup_context=_bce_setup)


def bce_with_logits(logits: Tensor, labels: Tensor) -> Tensor:
    """F.binary_cross_entropy_with_logits(logits, labels) (mean reduction, train.py:37) with its gradient made in the same pass:
    two launches for loss forward + backward instead of torch's chain."""
    return _bce_with_logits(logits, labels)[0]


# ------------------------------------------------------------------------------ SEAL / DGCNN (TwoWL/model/seal.py)


@torch.library.custom_op("twowl::seal_input", mutates_args=())
def seal_input(weight: Tensor, z: Tensor, feat: Optional[Tensor]) -> Tensor:
    """The first GCNConv's linear map of [one_hot(z, L) | feat] by weight [C, L + F] (L = weight.shape[1] - F, z in [0, L)): the
    feature product, then the columns weight[:, z] added by a gather (no one-hot matrix)."""
    L = weight.shape[1] - (0 if feat is None else feat.shape[1])
    if feat is None:
        return ops.label_gather(weight, z)
    out = ops.linear_fwd(_pad4(feat), _pad4(weight[:, L:]))
    return ops.label_gather(weight, z, out=out)


@seal_input.register_fake
def _(weight, z, feat):
    return weight.new_empty((z.numel(), weight.shape[0]))


def _si_setup(ctx, inputs, output):
    weight, z, feat = inputs
    ctx.save_for_backward(z, feat)
    ctx.L = weight.shape[1] - (0 if feat is None else feat.shape[1])


def _si_bwd(ctx, g):
    z, feat = ctx.saved_tensors
    g = g.contiguous()
    # d weight[:, l] = sum of g over the nodes labelled l: a segmented sum over the nodes grouped by label
    ptr, ids = ops.csr_build(z, ctx.L)
    dW = ops.seg_reduce(ptr, ids, ctx.L, g, plan=ops.seg_plan(ptr, ctx.L, ids.numel())).t()
    if feat is not None:
        dW = torch.cat((dW, ops.linear_bwd_weight(g, _pad4(feat))[:, :feat.shape[1]]), dim=1)
    return dW.contiguous(), None, None


seal_input.register_autograd(_si_bwd, setup_context=_si_setup)


@torch.library.custom_op("twowl::seal_tanh", mutates_args=())
def seal_tanh(h: Tensor) -> Tensor:
    return ops.tanh_slice_fwd(h, torch.empty_like(h), 0)


@seal_tanh.register_fake
def _(h):
    return torch.empty_like(h)


def _st_setup(ctx, inputs, output):
    ctx.save_for_backward(output)


def _st_bwd(ctx, g):
    (y,) = ctx.saved_tensors
    return ops.tanh_slice_bwd(g.contiguous(), y, 0, y.shape[1])


seal_tanh.register_autograd(_st_bwd, setup_context=_st_setup)


@torch.library.custom_op("twowl::seal_tanh_concat", mutates_args=())
def seal_tanh_concat(hs: List[Tensor], offs: List[int], width: int) -> Tensor:
    """[n, width]: tanh(hs[i]) in columns [offs[i], offs[i] + hs[i].shape[1]], zeros elsewhere (DGCNN's concatenated latents)."""
    out = hs[0].new_zeros((hs[0].shape[0], width))
    for h, off in zip(hs, offs):
        ops.tanh_slice_fwd(h, out, off)
    return out


@seal_tanh_concat.register_fake
def _(hs, offs, width):
    return hs[0].new_empty((hs[0].shape[0], width))


def _stc_setup(ctx, inputs, output):
    hs, offs, width = inputs
    ctx.save_for_backward(output)
    ctx.meta = [(off, h.shape[1]) for h, off in zip(hs, offs)]


def _stc_bwd(ctx, g):
    (y,) = ctx.saved_tensors
    g = g.contiguous()
    return [ops.tanh_slice_bwd(g, y, off, C) for off, C in ctx.meta], None, None


seal_tanh_concat.register_autograd(_stc_bwd, setup_context=_stc_setup)


@torch.library.custom_op("twowl::sort_pool", mutates_args=())
def sort_pool(x: Tensor, gptr: Tensor, k: int, key_col: int) -> Tuple[Tensor, Tensor]:
    """PyG global_sort_pool with ties broken by row -> (out [B, k, D], idx int32 [B, k]); only out is differentiable."""
    return ops.sortpool_fwd(x, gptr, k, key_col)


@sort_pool.register_fake
def _(x, gptr, k, key_col):
    B = gptr.shape[0] - 1
    return x.new_empty((B, k, x.shape[1])), x.new_empty((B, k), dtype=torch.int32)


def _sp_setup(ctx, inputs, output):
    ctx.save_for_backward(output[1])
    ctx.n_rows = inputs[0].shape[0]
    ctx.mark_non_differentiable(output[1])
    ctx.set_materialize_grads(False)


def _sp_bwd(ctx, g, _g_idx):
    (idx,) = ctx.saved_tensors
    return ops.sortpool_bwd(g, idx, ctx.n_rows), None, None, None


sort_pool.register_autograd(_sp_bwd, setup_context=_sp_setup)


@torch.library.custom_op("twowl::bias_act", mutates_args=())
def bias_act(y: Tensor, bias: Tensor, B: int, pool: int, relu: bool, p_drop: float, seed: int) -> Tensor:
    """ops.bias_act_fwd: bias + ReLU (optional) + max-pool over `pool` rows + dropout, y [B * Lin, C]."""
    return ops.bias_act_fwd(y, bias, B, pool, relu, p_drop, seed)


@bias_act.register_fake
def _(y, bias, B, pool, relu, p_drop, seed):
    return y.new_empty((B * ((y.shape[0] // max(B, 1)) // pool), y.shape[1]))


def _ba_setup(ctx, inputs, output):
    y, bias, B, pool, relu, p_drop, seed = inputs
    ctx.save_for_backward(y, bias)
    ctx.meta = (B, pool, relu, p_drop, seed)


def _ba_bwd(ctx, g):
    y, bias = ctx.saved_tensors
    dy = ops.bias_act_bwd(g, y, bias, *ctx.meta)
    return dy, ops.colsum(dy), None, None, None, None, None


bias_act.register_autograd(_ba_bwd, setup_context=_ba_setup)


@torch.library.custom_op("twowl::im2col", mutates_args=())
def im2col(p: Tensor, B: int, kw: int) -> Tensor:
    """ops.im2col_fwd: Conv1d's input windows as rows, p [B * L1, C] -> [B * (L1 - kw + 1), C * kw]."""
    return ops.im2col_fwd(p, B, kw)


@im2col.register_fake
def _(p, B, kw):
    L1 = p.shape[0] // B
    return p.new_empty((B * (L1 - kw + 1), p.shape[1] * kw))


def _i2c_setup(ctx, inputs, output):
    p, B, kw = inputs
    ctx.meta = (B, p.shape[0] // B, p.shape[1], kw)


def _i2c_bwd(ctx, g):
    return ops.im2col_bwd(g, *ctx.meta), None, None


im2col.register_autograd(_i2c_bwd, setup_context=_i2c_setup)
