"""Device-side index structures the kernels consume, built once per index tensor and cached.

The reference rebuilds gcn_norm (self-loop surgery + degree + edge weights) inside every GCNConv
call - depth1 + 2*depth2 times per forward (SURVEY.md K9). Here each index tensor is turned ONCE
into CSR-by-target (forward) and CSR-by-source (backward) plus its dinv vector, keyed by the
tensor's storage and version counter.
"""
from __future__ import annotations

from collections import OrderedDict
from dataclasses import dataclass, field
from typing import Optional

import torch

from . import ops


class _Cache:
    """Tiny LRU keyed by (data_ptr, shape, strides, version). Entries keep the key tensor alive, so a
    data_ptr can never be recycled by the allocator while its entry exists."""

    def __init__(self, cap: int = 24):   # train / val / test splits x (node graph, pair table, regrouped view, its pair table, ...)
        self.cap = cap
        self.d: "OrderedDict[tuple, tuple]" = OrderedDict()

    @staticmethod
    def key(t: torch.Tensor, *extra):
        return (t.data_ptr(), tuple(t.shape), tuple(t.stride()), t._version, t.device.index) + extra

    def get(self, t: torch.Tensor, extra, build):
        k = self.key(t, *extra)
        hit = self.d.get(k)
        if hit is not None:
            self.d.move_to_end(k)
            return hit[1]
        val = build()
        self.d[k] = (t, val)
        while len(self.d) > self.cap:
            self.d.popitem(last=False)
        return val

    def clear(self):
        self.d.clear()


_cache = _Cache()
# structures built from tensors that a training loop may recreate every step (an untagged edge tensor, an explicit [2,T']
# wedge tensor): their own small cache, so that one entry per step can neither pin 24 steps' worth of index memory nor evict
# the dataset-lifetime entries above (pair tables, regrouped views, row-shard blocks)
_step_cache = _Cache(cap=4)


def clear_cache():
    _cache.clear()
    _step_cache.clear()


def _i64(t: torch.Tensor) -> torch.Tensor:
    return t if t.dtype == torch.int64 else t.to(torch.int64)


# ------------------------------------------------------------------------------ node-level graph (edge1)

@dataclass
class NodeGraph:
    n: int
    ptr: torch.Tensor    # CSR by target: rows = ei[1], col = ei[0]
    col: torch.Tensor
    tptr: torch.Tensor   # CSR by source: rows = ei[0], col = ei[1]
    tcol: torch.Tensor
    dinv: torch.Tensor   # (1 + in-degree without self-loops)^-1/2
    plan: torch.Tensor   # long-row plans (ops.seg_plan) of the two CSRs
    tplan: torch.Tensor
    ids: Optional[torch.Tensor] = None     # edge position of every CSR entry (by target / by source)
    tids: Optional[torch.Tensor] = None
    emask: Optional[torch.Tensor] = None   # uint8 per ENTRY: removed from the cached CSRs (sample_block)
    temask: Optional[torch.Tensor] = None


class MaskedEdges:
    """The edge tensor `ei[:, ~mask]` of sample_block (utils.py:62-63) WITHOUT materialising it: the whole graph's edges plus a
    uint8[E] mask of the removed ones. Accepted by GCNConv.forward in place of the int64 [2,E'] tensor; needed where the
    data-dependent size E' must not reach the host (CUDA-graph capture of the step, twowl_b200.graphed)."""

    def __init__(self, ei: torch.Tensor, mask: torch.Tensor):
        self.ei, self.mask = ei, mask

    @property
    def device(self):
        return self.ei.device


def node_graph(edge1, n: int, _base: bool = False) -> NodeGraph:
    """CSR by target / by source + gcn_norm degrees of an int64 [2,E] edge tensor, cached per tensor. An edge tensor that
    sample_block produced (utils.py:61-64: the whole graph minus the sampled edge ids) reuses the cached CSRs of the
    whole graph with a per-entry mask instead of sorting its E' edges again every step."""
    if isinstance(edge1, MaskedEdges):
        tag = (edge1.ei, edge1.mask)
    else:
        tag = getattr(edge1, "_twowl_edges", None)
        if tag is not None and not (tag[2] == edge1._version and tag[0].shape[1] >= edge1.shape[1]):
            tag = None
    if tag is not None:
        base = node_graph(tag[0], n, _base=True)
        emask, temask = ops.gather_u8(tag[1], base.ids), ops.gather_u8(tag[1], base.tids)
        return NodeGraph(n, base.ptr, base.col, base.tptr, base.tcol, ops.gcn_dinv_entries(base.ptr, base.col, n, emask),
                         base.plan, base.tplan, base.ids, base.tids, emask, temask)

    def build():
        ei = _i64(edge1)
        ptr, ids = ops.csr_build(ei[1], n)
        col = ops.gather_cols(ids, ei[0])
        tptr, tids = ops.csr_build(ei[0], n)
        tcol = ops.gather_cols(tids, ei[1])
        m = ei.shape[1]
        return NodeGraph(n, ptr, col, tptr, tcol, ops.gcn_dinv(ptr, col, n), ops.seg_plan(ptr, n, m),
                         ops.seg_plan(tptr, n, m), ids, tids)
    # the base graph of a sample_block result / MaskedEdges is a dataset tensor; a bare tensor may be a per-step one
    return (_cache if _base else _step_cache).get(edge1, ("node", n), build)


def simple_adjacency(ei: torch.Tensor, n: int):
    """(ptr, adj) of ops.simple_adjacency for an int64 [2,E] edge tensor - the undirected simple graph the link heuristics
    intersect - cached per tensor, so that several heuristics or tables over one split build it once."""
    def build():
        e = _i64(ei)
        return ops.simple_adjacency(e[0], e[1], n)
    return _cache.get(ei, ("simple", n), build)


# ------------------------------------------------------------------------------ pair table (pos)

@dataclass
class PairTable:
    n: int               # number of nodes the features have
    R: int
    src: torch.Tensor    # int32 [R]
    dst: torch.Tensor
    ptr_s: torch.Tensor  # pair rows grouped by src node
    ids_s: torch.Tensor
    ptr_d: torch.Tensor  # pair rows grouped by dst node
    ids_d: torch.Tensor
    plan_s: torch.Tensor
    plan_d: torch.Tensor
    mated: bool = False  # rows 2k / 2k+1 are (u,v) / (v,u): the doubled layout of utils.py:81-90


def pair_table(pos: torch.Tensor, n: int) -> PairTable:
    def build():
        p = _i64(pos)
        ptr_s, ids_s = ops.csr_build(p[:, 0], n)
        ptr_d, ids_d = ops.csr_build(p[:, 1], n)
        R = p.shape[0]
        mated = False
        if R > 0:   # ONE host read per pair table (cached): the endpoints' range, and whether the doubled layout holds
            lo_hi = torch.stack((p.min(), p.max()))
            if R % 2 == 0:
                q = p.reshape(R // 2, 2, 2)
                lo_hi = torch.cat((lo_hi, ((q[:, 0, 0] == q[:, 1, 1]) & (q[:, 0, 1] == q[:, 1, 0])).all().reshape(1).to(p.dtype)))
            vals = lo_hi.tolist()
            if vals[0] < 0 or vals[1] >= n:
                # x[pos[:, 0]] of model.py:75 raises IndexError in the reference; the gather kernels do no bounds checks
                raise IndexError(f"pos holds node ids in [{vals[0]}, {vals[1]}] but the features have {n} rows")
            mated = len(vals) == 3 and bool(vals[2])
        return PairTable(n, R, ops.narrow_i32(p[:, 0]), ops.narrow_i32(p[:, 1]), ptr_s, ids_s, ptr_d, ids_d,
                         ops.seg_plan(ptr_s, n, R), ops.seg_plan(ptr_d, n, R), mated)
    return _cache.get(pos, ("pos", n), build)


# ------------------------------------------------------------------------------ explicit wedge index (any ei2)

@dataclass
class ExplicitWedges:
    R: int
    ptr_b: torch.Tensor   # CSR by target pair b, col = source edge a
    col_b: torch.Tensor
    ptr_a: torch.Tensor   # CSR by source edge a, col = target pair b
    col_a: torch.Tensor
    dinv: tuple           # (dinv for edge2 = [a^1; b], dinv for edge2_r = [a; b^1])
    plan_b: torch.Tensor
    plan_a: torch.Tensor


def explicit_wedges(ei2: torch.Tensor, R: int) -> ExplicitWedges:
    """reverse() (utils.py:71-78) is never materialised: both directions read the same two CSRs with the
    id^1 flips folded into the kernel (flip / row_flip)."""
    if R % 2:
        raise RuntimeError("the pair table must have an even number of rows (ids 2k/2k+1 are mates, utils.py:81-90)")

    def build():
        e = _i64(ei2)
        ptr_b, ids_b = ops.csr_build(e[1], R)
        col_b = ops.gather_cols(ids_b, e[0])
        ptr_a, ids_a = ops.csr_build(e[0], R)
        col_a = ops.gather_cols(ids_a, e[1])
        d0 = ops.gcn_dinv(ptr_b, col_b, R, flip=1, row_flip=0)
        d1 = ops.gcn_dinv(ptr_b, col_b, R, flip=0, row_flip=1)
        T = e.shape[1]
        return ExplicitWedges(R, ptr_b, col_b, ptr_a, col_a, (d0, d1), ops.seg_plan(ptr_b, R, T), ops.seg_plan(ptr_a, R, T))
    return _step_cache.get(ei2, ("ei2", R), build)


# ------------------------------------------------------------------------------ structured wedge index

@dataclass
class WedgeStruct:
    """What get_ei2(n_node, pos_edge, pred_edge) joins, kept in factored form: the in-list of observed
    edges per node and the out-list of pair rows per node. ``blocked`` (uint8[E]) marks source edges
    removed by blockei2. T = sum_i cin(i)*cout(i) wedges are implied, never stored."""
    n_node: int
    E: int
    R: int
    src: torch.Tensor      # int32 [R]  pos[:,0] of every pair row
    dst_e: torch.Tensor    # int32 [E]  target node of every observed edge
    in_ptr: torch.Tensor   # int64 [n+1], in_ids int32: observed edge ids grouped by target node (ascending id)
    in_ids: torch.Tensor
    out_ptr: torch.Tensor  # int64 [n+1], out_ids int32: pair rows grouped by source node (ascending id)
    out_ids: torch.Tensor
    in_plan: torch.Tensor  # long-row plans of the two lists (hubs)
    out_plan: torch.Tensor
    blocked: Optional[torch.Tensor] = None
    _prep: Optional[tuple] = field(default=None, repr=False)

    def with_blocked(self, blocked: torch.Tensor) -> "WedgeStruct":
        if self.blocked is not None:
            blocked = torch.maximum(blocked, self.blocked)
        return WedgeStruct(self.n_node, self.E, self.R, self.src, self.dst_e, self.in_ptr, self.in_ids, self.out_ptr,
                           self.out_ids, self.in_plan, self.out_plan, blocked)

    def prepared(self):
        """(cnt[N], centre[2,R], dinv[2,R], selfw[2,R], bnode[2,R]) - per-row constants of both directions."""
        if self._prep is None:
            if self.E % 2 or self.R % 2:
                raise RuntimeError("structured wedge path needs the doubled layout (even E and R)")
            self._prep = ops.wedge_prepare(self.src, self.dst_e, self.E, self.R, self.n_node, self.blocked, self.in_ptr)
        return self._prep

    def num_wedges(self) -> int:
        """T' = sum over unblocked a of cout(dst(a)) - one host read."""
        cin = (self.in_ptr[1:] - self.in_ptr[:-1]) if self.blocked is None else self.prepared()[0][: self.n_node].to(torch.int64)
        cout = self.out_ptr[1:] - self.out_ptr[:-1]
        return int((cin * cout).sum().item())


def build_wedge_struct(n_node: int, pos_edge: torch.Tensor, pred_edge: torch.Tensor) -> WedgeStruct:
    pos_edge, pred_edge = _i64(pos_edge), _i64(pred_edge)
    E, P = pos_edge.shape[1], pred_edge.shape[1]
    src_all = torch.cat((pos_edge[0], pred_edge[0]))
    in_ptr, in_ids = ops.csr_build(pos_edge[1], n_node)
    out_ptr, out_ids = ops.csr_build(src_all, n_node)
    return WedgeStruct(int(n_node), E, E + P, ops.narrow_i32(src_all), ops.narrow_i32(pos_edge[1]), in_ptr, in_ids,
                       out_ptr, out_ids, ops.seg_plan(in_ptr, int(n_node), E), ops.seg_plan(out_ptr, int(n_node), E + P))


def wedges_match_table(struct: "WedgeStruct", pt: PairTable) -> bool:
    """Does the factored wedge index describe THIS pair table - pos = [pos_edge^T ; pred_edge^T], the layout of
    datasets.py:95-99 - so that the factorised kernels (which read the centre / target nodes from the index and the pair
    endpoints from the table) compute what the explicit [2,T] tensor says? One device comparison per (index, table), cached;
    a mismatch sends the model to the explicit path, which follows the tensor whatever it holds."""
    def build():
        if struct.R != pt.R or struct.n_node > pt.n:
            return (pt, False)
        same = torch.equal(struct.src, pt.src) and torch.equal(struct.dst_e, pt.dst[: struct.E])
        return (pt, bool(same))
    # keyed on BOTH tensors' identity (pointer, shape, strides, version); the entry holds struct.src (as its key tensor) and pt
    # (in its value), so neither address can be recycled for another table while the verdict is cached
    return _cache.get(struct.src, ("match",) + _Cache.key(pt.src), build)[1]


@dataclass
class LocalityView:
    """The same pair table with its PAIRS (rows 2k, 2k+1 together) regrouped by their higher-degree endpoint, observed edges
    and prediction pairs separately (rows < E stay < E). The order of pair rows is an internal matter of the model - only
    `idx` and the blocked-edge mask refer to row ids - and in this order the in-list / out-list of a hub node is one contiguous
    run of rows: the per-node gathers of the pair layer (SH, dS, pair-init backward) stream instead of hopping through DRAM, and
    half of pair_conv's gathered rows repeat the previous row's. Sums run over the same terms in a different order."""
    perm: torch.Tensor      # int32 [R]  new row -> old row
    newid: torch.Tensor     # int64 [R]  old row -> new row
    pos: torch.Tensor       # int64 [R,2] the regrouped pair table (original node ids: pair_init gathers x by them)
    struct: WedgeStruct     # built on the regrouped table (nothing blocked), its NODE ids compacted (see locality_view)


def locality_view(struct: WedgeStruct, pos: torch.Tensor) -> LocalityView:
    def build():
        p = _i64(pos)
        R, E, n = struct.R, struct.E, struct.n_node
        deg = torch.bincount(p[:, 0], minlength=n)
        parts = []
        for lo, hi in ((0, E), (E, R)):
            u, v = p[lo:hi:2, 0], p[lo:hi:2, 1]
            primary = torch.where(deg[u] >= deg[v], u, v)
            order = torch.sort(primary, stable=True).indices            # pairs of one primary endpoint together, original order inside
            parts.append((lo + torch.stack((2 * order, 2 * order + 1), dim=1)).reshape(-1))
        perm = torch.cat(parts)
        newid = torch.empty_like(perm)
        newid[perm] = torch.arange(R, device=perm.device)
        pos2 = p[perm].contiguous()
        # The per-node tables of the pair layer (in-list sums S, their gradients dS) only matter on nodes that HAVE observed
        # in-edges: S is zero elsewhere and dS is consumed through the target node of a live edge only. The wedge structure is
        # therefore built on compacted node ids (nodes with in-edges -> 0..n_act-1, every other node -> -1, which the index
        # kernels treat as "no such node"): R-MAT 1M/16M has 408 k isolated nodes, so the tables - and, row-sharded, their
        # all-reduces - shrink by 39 %. The pair table itself keeps the original ids.
        active = torch.bincount(p[:E, 1], minlength=n) > 0                           # nodes with observed in-edges
        nid = torch.where(active, torch.cumsum(active.to(torch.int64), 0) - 1, torch.full_like(deg, -1))
        n_act = max(int(active.sum().item()), 1)                                     # once per pair table (cached)
        cpos = nid[pos2]
        st = build_wedge_struct(n_act, cpos[:E].t().contiguous(), cpos[E:].t().contiguous())
        return LocalityView(perm.to(torch.int32), newid, pos2, st)
    return _cache.get(pos, ("locality", struct.E, struct.R, struct.n_node), build)


class WedgeIndex:
    """A wedge index that is NOT materialised (T = sum deg^2 reaches 6.5e10 on R-MAT 1M/16M - 1 TB as
    int64 [2,T]). Accepted wherever the drop-in API takes ``ei2``: sample_block, LocalWLNet.forward."""

    def __init__(self, struct: WedgeStruct):
        self.struct = struct

    @property
    def device(self):
        return self.struct.src.device

    def num_wedges(self) -> int:
        return self.struct.num_wedges()

    def materialize(self) -> torch.Tensor:
        from TwoWL.utils import _materialize
        return _materialize(self.struct)
