"""Row-block sharding of the pair table over several GPUs (SURVEY 8(e)): ONE TwoWL step cut over the ranks.

Pair level (model.py:75-83). Rank g owns a block of pair rows = its contiguous share of the observed pairs followed by its
contiguous share of the prediction pairs (blocks_of; even boundaries: rows 2k / 2k+1 are the two directions of one pair,
utils.py:81-90, and stay together), i.e. its rows of every [R, C] activation, the observed edges and the target links that fall
into the block. On the factorised wedge path a pair row only talks to the other rows through
per-NODE sums, so the exchange per pair layer is

    forward   all_reduce  SH_f, SH_r   [2, N, C] fp32      in-list sums of the pair layer (partial over the rank's edges)
              all_reduce  moments      [2, 2C]   fp64      GraphNorm column (sum, sum of squares) of both branches
              all_reduce  logits       [L]       fp32      every rank ends with the full [L, 1] output of model.py:83
    backward  all_reduce  colsums      [6, C]    fp64      GraphNorm-backward / readout column sums over the selected rows
                                                           ([4, C] over all rows for a layer that is not the last)
              all_reduce  dS_f, dS_r   [2, N, C] fp32      gradient of the per-node sums

(N here = the nodes that have observed in-edges: graph.locality_view compacts the node ids of the wedge structure) instead of
the all-gather / reduce-scatter of [R, C] an explicit wedge index would need. The tables are produced and summed one node range
at a time (reduce_in_chunks / work_cuts): the all-reduce of a range runs while the next one is gathered.

Node level (model.py:71-73). The node-level GCNConv aggregations - the only node-level work that is not a cheap streaming pass -
are cut into NODE blocks [g*B, (g+1)*B), B = ceil(N / world): a rank reduces the in-lists (forward) / out-lists (backward) of
its own nodes only (twowl_seg_args.row_begin / row_end on the whole graph's CSR) and the blocks are exchanged:

    forward   all_gather  conv output  [N, C]    fp32      per node layer
    backward  all_reduce  d(x)         [N, C]    fp32      once, in the pair-init backward (its block's part of dx), pipelined by
                                                           node range like the per-node tables: dx leaves it COMPLETE
              all_gather  d(z)         [N, C]    fp32      per node layer
              all_reduce  d(emb)       [V, C]    fp32      the embedding gradient, summed over node blocks

Everything else at node level (embedding lookup, GraphNorm, the [N, C] x [C, C] linear layers) is a streaming pass of a few
hundred MB and stays replicated. Gradient bookkeeping: upstream of the dx all-reduce every rank holds COMPLETE gradients, so the
parameter gradients made there (and every other gradient that is complete on all ranks after a reduction: GraphNorm / readout
column sums) are kept on rank 0 only - the caller's ONE all-reduce (sum) of the flat parameter gradients is then exact
(dist.allreduce_grads); gradients made from a rank's own rows stay partial and are summed by that same all-reduce.

No step of this path reads device data on the host: the target links of a block are selected by a mask (links outside the block
carry row id -1, which the readout kernels skip), not by a compaction whose size the host would have to know.

Every rank computes the same numbers as the single-GPU path up to the summation order of those reductions. Covers any
depth1 >= 1, depth2 >= 1 on the structured wedge path with the doubled pair layout and widths the tensor-core kernels take
(32 / 64 / 128). Dropout masks are keyed by the LOCAL row id: statistically the same as the single-GPU run, not the same bits
(parity tests run with dropout 0 / eval mode); the replicated node-level dropout draws the same host seeds on every rank
(seed every rank's torch generator alike).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Optional, Tuple

import torch
import torch.distributed as dist

from . import functional as F2
from . import graph as G
from . import ops


def block_of(R: int, rank: int, world: int) -> Tuple[int, int]:
    """[lo, hi) of rank's share of R rows cut into contiguous blocks of equal numbers of undirected pairs (even boundaries)."""
    if R % 2:
        raise ValueError("the pair table must have an even number of rows")
    pairs = R // 2
    return 2 * (pairs * rank // world), 2 * (pairs * (rank + 1) // world)


def blocks_of(E: int, R: int, rank: int, world: int) -> Tuple[Tuple[int, int], Tuple[int, int]]:
    """rank's block of the pair table = ([olo, ohi), [plo, phi)): its share of the OBSERVED pairs (rows < E) followed by its
    share of the PREDICTION pairs (rows >= E). The two kinds of rows cost differently - only observed edges feed the in-list
    sums, only they can be blocked - so a contiguous cut of [0, R) would give the first ranks all of that work (measured at
    world 8 on R-MAT 1M/16M: 15.4 ms of compute on the ranks holding observed edges against 12.6 ms on the others)."""
    if E % 2 or R % 2 or not 0 <= E <= R:
        raise ValueError("the pair table must hold E observed rows and R - E prediction rows, both even (doubled layout)")
    olo, ohi = block_of(E, rank, world)
    plo, phi = block_of(R - E, rank, world)
    return (olo, ohi), (E + plo, E + phi)


def take_ranges(t: torch.Tensor, ranges) -> torch.Tensor:
    """rows of t inside the block's two ranges, observed share first (a copy)."""
    (olo, ohi), (plo, phi) = ranges
    return torch.cat((t[olo:ohi], t[plo:phi]))


def work_cuts(ptr_global: torch.Tensor, ptr_local: torch.Tensor, M: int, K: int):
    """Cut the M rows of a CSR into K consecutive ranges of about equal work (entries + a per-row cost worth 4 entries):
    -> [(lo, hi, has_long)]. The bounds come from the WHOLE graph's CSR `ptr_global`, which every rank holds - they must be the
    same on all ranks (they size the collectives); has_long = this rank's own CSR `ptr_local` has rows longer than
    TWOWL_LONG_ROW entries inside the range (a range without them runs the row pass only: no empty launches of the long-row
    passes). Reads 2K numbers on the host: call it where the result is cached."""
    if K <= 1 or M <= 1:
        return [(0, M, True)]
    p = ptr_global[:M + 1]
    work = p + 4 * torch.arange(M + 1, device=p.device, dtype=p.dtype)
    targets = (work[M] * torch.arange(1, K, device=p.device, dtype=p.dtype)) // K
    inner = torch.searchsorted(work, targets).clamp_(0, M)
    q = ptr_local[:M + 1]
    is_long = ((q[1:] - q[:-1]) > ops.LONG_ROW).to(torch.int32)
    csum = torch.cat((is_long.new_zeros(1), torch.cumsum(is_long, 0)))
    bounds = [0] + inner.tolist() + [M]
    longs = csum[torch.tensor(bounds, device=p.device)].tolist()
    return [(bounds[k], bounds[k + 1], longs[k + 1] > longs[k]) for k in range(K)]


def node_block(N: int, rank: int, world: int) -> Tuple[int, int, int]:
    """(lo, hi, B): rank's node block [lo, hi) of equal-size blocks B = ceil(N / world) (the last ones may be short or empty)."""
    B = -(-N // world)
    return min(rank * B, N), min((rank + 1) * B, N), B


_last_shard = None


class RowShard:
    """Assign to ``LocalWLNet.row_shard`` to run forward / backward on this rank's block of pair rows (and node block)."""

    def __init__(self, group=None, rank: Optional[int] = None, world: Optional[int] = None, dry: bool = False):
        """dry = True (tools/rowshard_dry.py only): the collectives are accounted but NOT run - one rank's compute of a
        world-size-W step timed on a single device; the numbers it produces are partial sums, not results."""
        global _last_shard
        self.group = group
        self.dry = bool(dry)
        if rank is None:
            rank = dist.get_rank(group) if dist.is_initialized() else 0
            world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank, self.world = int(rank), int(world)
        self.nccl = dist.is_initialized() and dist.get_backend(group) == "nccl"
        self.log = {}            # collective name -> [calls, bytes] since construction
        self.steps = 0
        # node ranges of the pipelined table exchanges (8 GPUs, R-MAT 1M/16M: 2 ranges 18.5 ms per step, 4 ranges 19.1 ms - every
        # range is three more launches over short lists)
        self.chunks = 2
        _last_shard = self

    def _account(self, what: str, t: torch.Tensor):
        e = self.log.setdefault(what, [0, 0])
        e[0] += 1
        e[1] += t.numel() * t.element_size()

    def all_reduce(self, t: torch.Tensor, what: str = "all_reduce") -> torch.Tensor:
        if self.world > 1:
            self._account("all_reduce " + what, t)
            if self.dry:
                return t
            with ops._P("nccl_all_reduce", 2 * t.numel() * t.element_size()):
                dist.all_reduce(t, group=self.group)
        return t

    def all_reduce_async(self, t: torch.Tensor, what: str):
        """Start an all-reduce of a contiguous tensor on the communication stream (it waits for what the current stream has
        enqueued so far); kernels launched next on the current stream overlap it. -> handle with .wait() (a stream wait)."""
        if self.world == 1:
            return None
        self._account("all_reduce " + what, t)
        if self.dry:
            return None
        return dist.all_reduce(t, group=self.group, async_op=True)

    def reduce_in_chunks(self, cuts, produce, tensors, what: str):
        """A per-node table made by a row-range kernel and summed over the ranks, pipelined: `produce(lo, hi, has_long)` fills
        rows [lo, hi) of every tensor in `tensors` ([M, C] each); the all-reduce of a chunk runs on the communication stream
        while the next chunk is produced. `cuts` = work_cuts(...): node ranges of equal WORK, taken from the last (most nodes,
        largest exchange) to the first (the hubs: fewest nodes), so that the one exchange nothing overlaps is the smallest."""
        handles = []
        for lo, hi, has_long in reversed(cuts):
            if hi <= lo:
                continue
            produce(lo, hi, has_long)
            for t in tensors:
                h = self.all_reduce_async(t[lo:hi], what)
                if h is not None:
                    handles.append(h)
        with ops._P("nccl_all_reduce_wait", 0):
            for h in handles:
                h.wait()

    def all_gather_blocks(self, full: torch.Tensor, B: int, what: str = "all_gather") -> torch.Tensor:
        """full: [world * B, C] whose block [rank*B, (rank+1)*B) this rank has filled -> every block filled, in place."""
        if self.world > 1:
            self._account("all_gather " + what, full)
            if self.dry:
                return full
            mine = full[self.rank * B:(self.rank + 1) * B]
            with ops._P("nccl_all_gather", full.numel() * full.element_size()):
                if self.nccl:
                    dist.all_gather_into_tensor(full, mine, group=self.group)     # in place: input = this rank's slice of output
                else:   # gloo (the CPU / single-device tests): blocks of the other ranks zeroed, then a sum
                    full[:self.rank * B].zero_()
                    full[(self.rank + 1) * B:].zero_()
                    dist.all_reduce(full, group=self.group)
        return full


def comm_summary():
    """Collectives of the most recent RowShard per step: {name: {"calls_per_step", "MB_per_step"}} (bench.py)."""
    s = _last_shard
    if s is None or not s.steps:
        return None
    out = {k: {"calls_per_step": round(v[0] / s.steps, 2), "MB_per_step": round(v[1] / s.steps / 1e6, 2)} for k, v in sorted(s.log.items())}
    out["total_MB_per_step"] = round(sum(v[1] for v in s.log.values()) / s.steps / 1e6, 1)
    return out


# ------------------------------------------------------------------------------ node level


class _Rank0Grad(torch.autograd.Function):
    """Identity on a parameter whose gradient is COMPLETE on every rank: keep it on rank 0 so that the caller's sum is exact."""

    @staticmethod
    def forward(ctx, p, shard):
        ctx.keep = shard.rank == 0
        return p.view_as(p)

    @staticmethod
    def backward(ctx, g):
        return (g if ctx.keep else torch.zeros_like(g)), None


class _ShardedEmbedding(torch.autograd.Function):
    """nn.Embedding lookup by degree (model.py:71), replicated; backward = the segmented row sum by degree over this rank's
    NODE block of a gradient that is complete on every rank, summed over the ranks, kept on rank 0."""

    @staticmethod
    def forward(ctx, weight, deg, shard):
        ctx.save_for_backward(deg)
        ctx.meta = (weight.shape[0], shard)
        return ops.gather_rows(weight.contiguous(), deg)

    @staticmethod
    def backward(ctx, g):
        (deg,) = ctx.saved_tensors
        V, shard = ctx.meta
        deg = deg.reshape(-1)
        lo, hi, _ = node_block(deg.numel(), shard.rank, shard.world)
        g = g.contiguous()
        if hi > lo:
            ptr, ids = ops.csr_build(deg[lo:hi], V)     # rows = degree values: extremely skewed, so plan it
            plan = ops.seg_plan(ptr, V, hi - lo)
            dW = ops.seg_reduce(ptr, ids, V, g[lo:hi], plan=plan)
        else:
            dW = g.new_zeros((V, g.shape[1]))
        shard.all_reduce(dW, "d(emb) [V,C]")
        if shard.rank != 0:
            dW.zero_()
        return dW, None, None


class _ShardedNodeAggregate(torch.autograd.Function):
    """GCNConv.propagate + bias of a node layer (model.py:73; functional.gcn_aggregate) with the output rows cut into node blocks:
    this rank reduces the in-lists of its own nodes and the blocks are all-gathered. Backward: the out-lists of the rank's own
    nodes, all-gather -> d(z) complete on every rank; d(bias) complete, kept on rank 0. (grad_is_partial=True first sums an
    incoming gradient that is still partial over the ranks; the pair level now hands back a complete dx, so forward_nodes
    passes False.)"""

    @staticmethod
    def forward(ctx, z, bias, gr, shard, grad_is_partial):
        z = z.contiguous()
        N, C = z.shape
        lo, hi, B = node_block(N, shard.rank, shard.world)
        full = torch.empty((B * shard.world, C), dtype=z.dtype, device=z.device)
        ops.seg_reduce(gr.ptr, gr.col, N, z, plan=gr.plan, src_scale=gr.dinv, dst_scale=gr.dinv, skip_self=True, self_mode=1, bias=bias,
                       entry_mask=gr.emask, out=full[:N], rows=(lo, hi))
        shard.all_gather_blocks(full, B, "node conv out [N,C]")
        ctx.gr, ctx.shard, ctx.partial = gr, shard, bool(grad_is_partial)
        return full[:N]

    @staticmethod
    def backward(ctx, g):
        gr, shard = ctx.gr, ctx.shard
        N, C = g.shape
        lo, hi, B = node_block(N, shard.rank, shard.world)
        if ctx.partial:
            g = shard.all_reduce(g.clone(memory_format=torch.contiguous_format), "d(x) [N,C]")
        else:
            g = g.contiguous()
        dbias = ops.colsum(g) if shard.rank == 0 else g.new_zeros((C,))
        full = torch.empty((B * shard.world, C), dtype=g.dtype, device=g.device)
        ops.seg_reduce(gr.tptr, gr.tcol, N, g, plan=gr.tplan, src_scale=gr.dinv, dst_scale=gr.dinv, skip_self=True, self_mode=1,
                       entry_mask=gr.temask, out=full[:N], rows=(lo, hi))
        shard.all_gather_blocks(full, B, "node d(z) [N,C]")
        return full[:N], dbias, None, None, None


class _NodeLinear(torch.autograd.Function):
    """z = h W^T of a node layer, replicated (a streaming pass). Its input gradient is complete on every rank; the weight gradient
    dz^T h runs over the N nodes, so every rank takes its node block and the caller's gradient sum completes it."""

    @staticmethod
    def forward(ctx, h, w, shard):
        h = h.contiguous()
        ctx.save_for_backward(h, w)
        ctx.shard = shard
        return ops.linear_fwd(h, w.contiguous())

    @staticmethod
    def backward(ctx, g):
        h, w = ctx.saved_tensors
        shard = ctx.shard
        g = g.contiguous()
        lo, hi, _ = node_block(h.shape[0], shard.rank, shard.world)
        dh = ops.linear_bwd_input(g, w.contiguous()) if ctx.needs_input_grad[0] else None
        dw = ops.linear_bwd_weight(g[lo:hi], h[lo:hi]) if hi > lo else torch.zeros_like(w)
        return dh, dw, None


def node_graph_block(edge1, N: int, shard: "RowShard") -> G.NodeGraph:
    """graph.node_graph for ONE rank of a row-sharded step. The node graph of a step is the cached CSR of the whole graph minus
    the edges sample_block took out (a per-entry mask) with the gcn_norm degrees recounted - E-sized work per step that every
    rank would repeat (0.77 ms at R-MAT 1M/16M: two mask gathers + the degree count). A rank only ever reduces the lists of its
    own node block, so it carries the mask to the entries of ITS block's rows in the two CSRs and counts ITS nodes' degrees; the
    blocks of dinv (N floats) are all-gathered. Everything outside the block's entry ranges of emask / temask is unset and never
    read (seg_reduce with rows = the block). Any other edge tensor takes the replicated graph.node_graph."""
    if isinstance(edge1, G.MaskedEdges):
        tag = (edge1.ei, edge1.mask)
    else:
        tag = getattr(edge1, "_twowl_edges", None)
        if tag is not None and not (tag[2] == edge1._version and tag[0].shape[1] >= edge1.shape[1]):
            tag = None
    if tag is None or shard.world == 1:
        return G.node_graph(edge1, N)
    base = G.node_graph(tag[0], N, _base=True)
    lo, hi, B = node_block(N, shard.rank, shard.world)
    # entry ranges of the block's rows in the two CSRs: four numbers read once per whole graph and rank (cached with it)
    e0, e1, t0, t1 = G._cache.get(base.ptr, ("rowshard-node-entries", lo, hi),
                                  lambda: tuple(int(v) for v in torch.stack((base.ptr[lo], base.ptr[hi], base.tptr[lo], base.tptr[hi])).tolist()))
    emask = torch.empty(base.ids.numel(), dtype=torch.uint8, device=base.ids.device)
    temask = torch.empty(base.tids.numel(), dtype=torch.uint8, device=base.ids.device)
    if e1 > e0:
        ops.gather_u8(tag[1], base.ids[e0:e1], out=emask[e0:e1])
    if t1 > t0:
        ops.gather_u8(tag[1], base.tids[t0:t1], out=temask[t0:t1])
    dinv = torch.empty(B * shard.world, dtype=torch.float32, device=base.ids.device)
    ops.gcn_dinv_entries(base.ptr, base.col, N, emask, rows=(lo, hi), out=dinv)
    shard.all_gather_blocks(dinv.view(-1, 1), B, "node dinv [N]")
    return G.NodeGraph(N, base.ptr, base.col, base.tptr, base.tcol, dinv[:N], base.plan, base.tplan, base.ids, base.tids, emask, temask)


def forward_nodes(model, x, edge1):
    """model.py:71-73 with the aggregations cut into node blocks: x int64 [N] degrees -> [N, C] (complete on every rank)."""
    shard: RowShard = model.row_shard
    if model.use_node_feat:
        raise NotImplementedError("row sharding covers the degree-embedding input (use_node_feat=False)")
    N = x.numel()

    def r0(p):
        return _Rank0Grad.apply(p, shard)

    def gn_act(gn, dp, act, h):
        p = dp.p if (model.training and dp.p > 0.0) else 0.0
        seed = ops.next_seed() if p > 0.0 else 0
        return F2.graphnorm_act(h, r0(gn.weight), r0(gn.bias), r0(gn.mean_scale), None, gn.eps, p, seed, isinstance(act, torch.nn.ReLU))[0]

    emb, gn0, dp0 = model.emb[0], model.emb[1], model.emb[2]
    h = _ShardedEmbedding.apply(emb.weight, x, shard)
    h = gn_act(gn0, dp0, None, h)
    gr = None
    for k, seq in enumerate(model.conv1s):
        conv, gn, dp, act = seq.modlist[0], seq.modlist[1], seq.modlist[2], seq.modlist[3]
        gr = gr if gr is not None else node_graph_block(edge1, N, shard)
        z = _NodeLinear.apply(h, conv.lin.weight, shard)
        out = _ShardedNodeAggregate.apply(z, conv.bias, gr, shard, False)
        h = gn_act(gn, dp, act, out)      # the pair level hands back a COMPLETE dx (summed in _ShardedPairInit.backward)
    return h


# ------------------------------------------------------------------------------ pair level


@dataclass
class _Local:
    ranges: tuple          # ((olo, ohi), (plo, phi)) rows of the table this block holds, in this order
    E_loc: int             # observed edges inside the block (its first ohi - olo rows)
    src: torch.Tensor      # int32 [Rl]
    dst: torch.Tensor
    in_ptr: torch.Tensor   # the block's observed edges grouped by target node (local ids)
    in_ids: torch.Tensor
    in_plan: torch.Tensor
    out_ptr: torch.Tensor  # the block's pair rows grouped by source node (local ids), in the wedge structure's node ids
    out_ids: torch.Tensor
    out_plan: torch.Tensor
    xout_ptr: torch.Tensor  # the same grouping by the pair TABLE's (original) node ids = pair_init's backward CSR
    xout_ids: torch.Tensor
    xout_plan: torch.Tensor
    in_cuts: list           # work_cuts of the three CSRs: node ranges of the pipelined table exchanges
    out_cuts: list
    xout_cuts: list


def _local(struct: G.WedgeStruct, pt: G.PairTable, ranges, K: int = 1) -> _Local:
    (olo, ohi), (plo, phi) = ranges

    def build():
        n = struct.n_node
        El, Rl = ohi - olo, (ohi - olo) + (phi - plo)
        src_l, dst_l = take_ranges(pt.src, ranges), take_ranges(pt.dst, ranges)
        in_ptr, in_ids = ops.csr_build(struct.dst_e[olo:ohi].to(torch.int64), n)
        out_ptr, out_ids = ops.csr_build(take_ranges(struct.src, ranges).to(torch.int64), n)
        xout_ptr, xout_ids = ops.csr_build(src_l.to(torch.int64), pt.n)
        return (pt, _Local(ranges, El, src_l, dst_l, in_ptr, in_ids, ops.seg_plan(in_ptr, n, El), out_ptr, out_ids,
                           ops.seg_plan(out_ptr, n, Rl), xout_ptr, xout_ids, ops.seg_plan(xout_ptr, pt.n, Rl),
                           work_cuts(struct.in_ptr, in_ptr, n, K), work_cuts(struct.out_ptr, out_ptr, n, K),
                           work_cuts(pt.ptr_s, xout_ptr, pt.n, K)))
    # the entry holds struct.src (key tensor) and pt (value): neither address can be recycled while the block is cached
    return G._cache.get(struct.src, ("rowshard", olo, ohi, plo, phi, K) + G._Cache.key(pt.src), build)[1]


def _layer_forward(shard, loc, rows, blocked_l, R_total, n_node, eps, H, pf, pr):
    """Both directions' pre-GraphNorm outputs of one pair layer on this block + the GLOBAL statistics:
    -> (O_f, O_r, stats_f, stats_r, SH [2,N,C])."""
    centre, dinv, selfw, _ = rows
    (wf, bf, gmf), (wr, br, gmr) = pf, pr
    # both directions' in-list sums (SH[0] = forward, SH[1] = reverse) from one pass over the block's edges, produced one node
    # range at a time so that the all-reduce of a range overlaps the gathers of the next
    SH = torch.empty((2, n_node, H.shape[1]), dtype=H.dtype, device=H.device)
    shard.reduce_in_chunks(loc.in_cuts,
                           lambda lo, hi, lg: ops.seg_reduce(loc.in_ptr, loc.in_ids, n_node, H, plan=loc.in_plan if lg else None,
                                                             src_scale=dinv[1], skip_mask=blocked_l, dual=True, src_scale2=dinv[0],
                                                             out=SH[1], out2=SH[0], rows=(lo, hi)),
                           (SH[0], SH[1]), "SH [2,N,C]")
    Sf, Sr = ops.linear_fwd(SH[0], wf), ops.linear_fwd(SH[1], wr)
    Os, moms = [], []
    for d, (w, b, gm, S) in enumerate(((wf, bf, gmf, Sf), (wr, br, gmr, Sr))):
        O, mom = ops.pair_conv([H], [w], [0], row_scale=[selfw[d]], gathers=[(S, centre[d], dinv[d])], bias=b,
                               stats_mean_scale=gm, eps=eps, want_moments=True)
        Os.append(O)
        moms.append(mom)
    mom = shard.all_reduce(torch.stack(moms), "GraphNorm moments [2,2C] f64")
    sf = ops.graphnorm_stats_from_moments(mom[0], R_total, gmf, eps)
    sr = ops.graphnorm_stats_from_moments(mom[1], R_total, gmr, eps)
    return Os[0], Os[1], sf, sr, SH


def _layer_backward(shard, loc, rows, n_node, H, wf, wr, SH, dOf, dOr, dWf, dWr, pair_sum_out=False):
    """From the gradients of the two pre-GraphNorm outputs (and the (selfw*dO)^T H parts of the weight gradients) to
    (dH, dW_f, dW_r) on this block: the dS exchange and the input-gradient pass."""
    _, dinv, selfw, bnode = rows
    dOs = (dOf, dOr)
    dS = torch.empty((2, n_node, H.shape[1]), dtype=H.dtype, device=H.device)
    dOf_c, dOr_c = dOs[0].contiguous(), dOs[1].contiguous()
    shard.reduce_in_chunks(loc.out_cuts,
                           lambda lo, hi, lg: ops.seg_reduce(loc.out_ptr, loc.out_ids, n_node, dOf_c, plan=loc.out_plan if lg else None,
                                                             src_scale=dinv[0], dual=True, src_scale2=dinv[1], X_mate=dOr_c,
                                                             out=dS[0], out2=dS[1], rows=(lo, hi)),
                           (dS[0], dS[1]), "dS [2,N,C]")
    # dW_d = (selfw_d * dO_d)^T H + dS_d^T SH_d: the second product runs over the N nodes - every rank takes its NODE block of
    # the (now complete) dS and SH, and the caller's gradient sum over the ranks completes the product
    lo, hi, _ = node_block(n_node, shard.rank, shard.world)
    if hi > lo:
        dWf = dWf + ops.linear_bwd_weight(dS[0, lo:hi], SH[0, lo:hi])
        dWr = dWr + ops.linear_bwd_weight(dS[1, lo:hi], SH[1, lo:hi])
    dSW = [ops.linear_bwd_input(dS[0], wf), ops.linear_bwd_input(dS[1], wr)]
    # pair_sum_out: dh is [Rl / 2, C], dH[2k] + dH[2k+1] per pair - all the pair-init backward reads (functional.pair_init_layer_readout)
    dh = ops.pair_conv([dOf, dOr], [wf, wr], [1, 1], row_scale=[selfw[0], selfw[1]],
                       gathers=[(dSW[0], bnode[0], dinv[0]), (dSW[1], bnode[1], dinv[1])], pair_sum_out=pair_sum_out)
    return dh, dWf, dWr


def _param_grads(shard, C, dpf, dpr, extra=()):
    """dparams = [d gn.weight | d gn.bias | d gn.mean_scale | d conv.bias], made from rank-summed column sums, i.e. complete on
    every rank: kept on rank 0 so that the caller's SUM over ranks is exact."""
    if shard.rank != 0:
        for t in (dpf, dpr) + tuple(extra):
            t.zero_()
    return (dpf[3 * C:], dpf[:C], dpf[C:2 * C], dpf[2 * C:3 * C]), (dpr[3 * C:], dpr[:C], dpr[C:2 * C], dpr[2 * C:3 * C])


class _ShardedPairInit(torch.autograd.Function):
    """model.py:75 on one row block: x [N, C] (replicated) -> H [Rl, C]; backward = this block's part of dx, summed over the
    ranks one node range at a time while the next range is gathered -> dx complete on every rank."""

    @staticmethod
    def forward(ctx, x, loc, shard):
        x = x.contiguous()
        ctx.save_for_backward(x)
        ctx.meta = (loc, shard)
        return ops.pair_init_fwd(x, loc.src, loc.dst)

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        loc, shard = ctx.meta
        g = g.contiguous()
        N = x.shape[0]
        dx = torch.empty_like(x)
        shard.reduce_in_chunks(loc.xout_cuts,
                               lambda lo, hi, lg: ops.seg_reduce(loc.xout_ptr, loc.xout_ids, N, g, plan=loc.xout_plan if lg else None, X2=x,
                                                                 mul_idx=loc.dst, pair_sum=True, out=dx, rows=(lo, hi)),
                               (dx,), "d(x) [N,C]")
        return dx, None, None


class _ShardedPairLayer(torch.autograd.Function):
    """A conv2s[i] / conv2s_r[i] layer that is NOT the last one (model.py:77) on one row block: H [Rl, C] -> H' [Rl, C]."""

    @staticmethod
    def forward(ctx, H, wf, bf, gwf, gbf, gmf, wr, br, gwr, gbr, gmr, shard, loc, rows, blocked_l, R_total, n_node, eps, p_drop,
                seed_f, seed_r):
        H = H.contiguous()
        Of, Or, sf, sr, SH = _layer_forward(shard, loc, rows, blocked_l, R_total, n_node, eps, H, (wf, bf, gmf), (wr, br, gmr))
        hn = ops.graphnorm_apply2(Of, Or, sf, sr, (gwf, gbf, gmf), (gwr, gbr, gmr), p_drop, seed_f, seed_r, True)
        ctx.save_for_backward(H, wf, gwf, gbf, gmf, wr, gwr, gbr, gmr, Of, Or, sf, sr, SH, *rows)
        ctx.meta = (shard, loc, R_total, n_node, p_drop, seed_f, seed_r)
        return hn

    @staticmethod
    def backward(ctx, g):
        H, wf, gwf, gbf, gmf, wr, gwr, gbr, gmr, Of, Or, sf, sr, SH, *rows = ctx.saved_tensors
        shard, loc, R_total, n_node, p_drop, seed_f, seed_r = ctx.meta
        C = wf.shape[0]
        dOf, dOr, dpf, dpr = ops.graphnorm_bwd2(Of, Or, g.contiguous(), sf, sr, (gwf, gbf, gmf), (gwr, gbr, gmr), p_drop, seed_f, seed_r,
                                                True, R_total, lambda t: shard.all_reduce(t, "GraphNorm-backward column sums [4,C] f64"))
        dWf, dWr = ops.pair_dw(dOf, dOr, rows[2][0], rows[2][1], H)
        dh, dWf, dWr = _layer_backward(shard, loc, rows, n_node, H, wf, wr, SH, dOf, dOr, dWf, dWr)
        gf, gr = _param_grads(shard, C, dpf, dpr)
        return (dh, dWf) + gf + (dWr,) + gr + (None,) * 10


class _ShardedLastLayer(torch.autograd.Function):
    """The last conv2s / conv2s_r layer (model.py:77) + readout (model.py:78-83) on one row block: H [Rl, C] -> [L, 1] with the
    logits of the target links inside the block and 0 for the others (idx_l = -1 there).
    init_inside (depth2 = 1): the first argument is the node features x [N, C]; the pair init (model.py:75) runs inside, and the
    backward returns dx: the input-gradient GEMM writes one row per pair and the pair-init backward - pipelined with the dx
    exchange as in _ShardedPairInit - reads that (functional.pair_init_layer_readout on one row block)."""

    @staticmethod
    def forward(ctx, H, wf, bf, gwf, gbf, gmf, wr, br, gwr, gbr, gmr, pw, pb, shard, loc, rows, idx_l, blocked_l, R_total, n_node,
                eps, p_drop, seed_f, seed_r, init_inside=False):
        H = H.contiguous()
        x = H if init_inside else H.new_empty(0)
        if init_inside:
            H = ops.pair_init_fwd(x, loc.src, loc.dst)
        Of, Or, sf, sr, SH = _layer_forward(shard, loc, rows, blocked_l, R_total, n_node, eps, H, (wf, bf, gmf), (wr, br, gmr))
        if idx_l.numel():
            pred = ops.gn2_readout_fwd(Of, Or, sf, sr, (gwf, gbf, gmf), (gwr, gbr, gmr), p_drop, seed_f, seed_r, True, idx_l,
                                       pw.contiguous(), pb)
        else:
            pred = H.new_empty((0, 1))
        ctx.save_for_backward(x, H, wf, gwf, gbf, gmf, wr, gwr, gbr, gmr, pw, idx_l, Of, Or, sf, sr, SH, *rows)
        ctx.meta = (shard, loc, R_total, n_node, p_drop, seed_f, seed_r, bool(init_inside))
        return pred

    @staticmethod
    def backward(ctx, g):
        x, H, wf, gwf, gbf, gmf, wr, gwr, gbr, gmr, pw, idx_l, Of, Or, sf, sr, SH, *rows = ctx.saved_tensors
        shard, loc, R_total, n_node, p_drop, seed_f, seed_r, init_inside = ctx.meta
        C = wf.shape[0]
        pf, pr = (gwf, gbf, gmf), (gwr, gbr, gmr)
        Gp, head, nxt, consts, dpf, dpr, dpw, dpb = ops.gn2_readout_bwd_prepare(
            Of, Or, sf, sr, pf, pr, p_drop, seed_f, seed_r, True, idx_l, pw.contiguous(), g.reshape(-1), R_total,
            lambda t: shard.all_reduce(t, "readout / GraphNorm-backward column sums [6,C] f64"))
        dOf, dOr, dWf, dWr = ops.pair_dw_gn(Of, Or, consts, Gp, head, nxt, p_drop, seed_f, seed_r, True, rows[2][0], rows[2][1], H)
        dh, dWf, dWr = _layer_backward(shard, loc, rows, n_node, H, wf, wr, SH, dOf, dOr, dWf, dWr, pair_sum_out=init_inside)
        if init_inside:      # dh holds one row per pair: this block's part of dx from it, summed over the ranks range by range
            N, dh2 = x.shape[0], dh
            dh = torch.empty_like(x)
            shard.reduce_in_chunks(loc.xout_cuts,
                                   lambda lo, hi, lg: ops.seg_reduce(loc.xout_ptr, loc.xout_ids, N, dh2, plan=loc.xout_plan if lg else None,
                                                                     X2=x, mul_idx=loc.dst, x_pairs=True, out=dh, rows=(lo, hi)),
                                   (dh,), "d(x) [N,C]")
        gf, gr = _param_grads(shard, C, dpf, dpr, extra=(dpw, dpb))
        return (dh, dWf) + gf + (dWr,) + gr + (dpw.reshape(pw.shape), dpb) + (None,) * 12


class _SumLogits(torch.autograd.Function):
    """Every rank's [L, 1] logits (its own links filled, 0 elsewhere) -> the full [L, 1] tensor of model.py:83 on every rank (one
    all-reduce of L floats). Backward: the whole gradient to every rank - the masked readout backward uses its own links' only."""

    @staticmethod
    def forward(ctx, pred_l, shard):
        return shard.all_reduce(pred_l.clone(), "logits [L]")

    @staticmethod
    def backward(ctx, g):
        return g, None


def supported(model, wedges, C: int) -> Optional[str]:
    """None if the sharded path covers this model / input, else the reason."""
    if len(model.conv2s) < 1:
        return "row sharding needs at least one pair layer"
    if not isinstance(wedges, G.WedgeStruct):
        return "row sharding needs the structured wedge index (TwoWL.utils.get_ei2 / sample_block)"
    if not all(F2.pair_layer_supported(wedges, C, f, r) for f, r in zip(model.conv2s, model.conv2s_r)) or not ops.pair_dw_supported(C):
        return f"pair width {C} is not covered by the tensor-core pair kernels"
    return None


def mask_links(idx: torch.Tensor, ranges) -> torch.Tensor:
    """Readout row ids [2L] -> block-local ids for the rows inside the block's two ranges (observed share first, then the
    prediction share), -1 for the others; both rows of a link are the two directions of one pair (double(.., for_index=True)),
    so they are inside or outside together (asserted on the device)."""
    (olo, ohi), (plo, phi) = ranges
    in_o = (idx >= olo) & (idx < ohi)
    in_p = (idx >= plo) & (idx < phi)
    inb = in_o | in_p
    torch._assert_async((inb[0::2] == inb[1::2]).all(),
                        "row-sharded readout: idx[2l] and idx[2l+1] must be the two rows of one pair (double(.., for_index=True))")
    return torch.where(in_o, idx - olo, torch.where(in_p, idx - (plo - (ohi - olo)), torch.full_like(idx, -1)))


MASKED_TAIL = -2     # readout row id: this link and every later one is masked (include/twowl.h, twowl_gn2_readout_fwd)


def own_links_first(idx_l: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """Masked readout ids [2L] -> (the same links stably partitioned: this rank's first, the masked ones after them; dest [L] =
    new position of link l). The readout kernels skip a masked link, but one lane group then meets its own links one at a
    time between skipped ones and waits out a full gather latency for each (ncu, world 8: 0.36 + 0.65 ms at 1.2 TB/s for an
    eighth of the links); with the rank's links packed at the front the groups work on them side by side, and the masked
    links behind them carry the id MASKED_TAIL, at which the kernels stop. No size reaches the host: the count of own links stays a device scalar inside `dest`."""
    L = idx_l.numel() // 2
    valid = idx_l[0::2] >= 0
    cv = torch.cumsum(valid, 0)
    pos = torch.arange(L, device=idx_l.device)
    dest = torch.where(valid, cv - 1, cv[-1] + (pos - cv))
    packed = torch.empty_like(idx_l).view(L, 2)
    packed[dest] = torch.where(valid.unsqueeze(1), idx_l.view(L, 2), torch.full_like(idx_l.view(L, 2), MASKED_TAIL))
    return packed.view(-1), dest


def forward(model, x, edge1, pos, idx, ei2):
    """LocalWLNet.forward (model.py:68-84) cut over the ranks: node blocks for the node-level aggregations, row blocks of the pair
    table for the pair level; returns the full [L, 1] logits on every rank."""
    model.row_shard.steps += 1
    return forward_pairs(model, forward_nodes(model, x, edge1), pos, idx, ei2)


def forward_pairs(model, x, pos, idx, ei2):
    """The pair-level part of LocalWLNet.forward (model.py:75-83) on this rank's row block; returns the full [L, 1] logits."""
    shard: RowShard = model.row_shard
    if idx is None:
        raise RuntimeError("row-sharded forward needs idx (the target links)")
    pt = G.pair_table(pos, x.shape[0])
    wedges = model._wedges(ei2, pt.R, pt)
    why = supported(model, wedges, x.shape[1])
    if why is None and not pt.mated:
        why = "row sharding needs the doubled pair layout (rows 2k / 2k+1 = (u,v) / (v,u))"
    if why is not None:
        raise NotImplementedError(why)
    idx = ops.index_guard(idx, pt.R, "idx")      # x[idx] of model.py:78: negative ids wrap, anything else out of range asserts
    if getattr(model, "pair_locality", False):
        # the blocks are cut from the pair table regrouped by hub (graph.LocalityView): same rows, streaming per-node gathers
        lv = G.locality_view(wedges, pos)
        pt = G.pair_table(lv.pos, x.shape[0])
        blocked = wedges.blocked
        wedges = lv.struct if blocked is None else lv.struct.with_blocked(ops.gather_u8(blocked, lv.perm[:wedges.E]))
        idx = lv.newid[idx]
    ranges = blocks_of(wedges.E, pt.R, shard.rank, shard.world)
    loc = _local(wedges, pt, ranges, shard.chunks if shard.world > 1 else 1)
    # per-row constants of THIS block only (the degree counts are global: every rank holds the int edge lists)
    _, centre, dinv, selfw, bnode = ops.wedge_prepare(wedges.src, wedges.dst_e, wedges.E, wedges.R, wedges.n_node, wedges.blocked,
                                                      wedges.in_ptr, ranges)
    rows = (centre, dinv, selfw, bnode)
    blocked_l = wedges.blocked[ranges[0][0]:ranges[0][1]] if wedges.blocked is not None else None
    idx_l, link_dest = own_links_first(mask_links(idx, ranges))
    last = len(model.conv2s) - 1
    init_inside = last == 0 and getattr(model, "fused_pair_init", True)      # depth2 = 1: the pair init joins the last layer's node
    H = x if init_inside else _ShardedPairInit.apply(x, loc, shard)
    for i, (seq_f, seq_r) in enumerate(zip(model.conv2s, model.conv2s_r)):
        cf, gf, dpf = seq_f.modlist[0], seq_f.modlist[1], seq_f.modlist[2]
        cr, gr = seq_r.modlist[0], seq_r.modlist[1]
        p = dpf.p if (model.training and dpf.p > 0.0) else 0.0
        seeds = [ops.next_seed() for _ in range(2)] if p > 0.0 else [0, 0]
        par = (cf.lin.weight, cf.bias, gf.weight, gf.bias, gf.mean_scale, cr.lin.weight, cr.bias, gr.weight, gr.bias, gr.mean_scale)
        if i < last:
            H = _ShardedPairLayer.apply(H, *par, shard, loc, rows, blocked_l, pt.R, wedges.n_node, gf.eps, p, seeds[0], seeds[1])
        else:
            pred_l = _ShardedLastLayer.apply(H, *par, model.pred.weight, model.pred.bias, shard, loc, rows, idx_l, blocked_l, pt.R,
                                             wedges.n_node, gf.eps, p, seeds[0], seeds[1], init_inside)
    return _SumLogits.apply(pred_l.index_select(0, link_dest), shard)       # back to the caller's link order
