"""Tensor-level wrappers over the C ABI (include/twowl.h): allocate outputs and workspaces with
the PyTorch caching allocator, pass raw device pointers and the current CUDA stream.

Nothing here computes on the host and nothing falls back to torch ops: a CPU tensor raises.
Data-dependent sizes (T of get_ei2, T' of blockei2) cost one device->host scalar read each,
exactly where the reference's own torch ops (cat / boolean indexing) synchronise.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional, Tuple

import numpy as np
import torch

from ._lib import ConvArgs, SegArgs, check, lib

SELECT_TILE = 2048
_launches = 0  # number of C-ABI compute calls issued (bench.py reports kernels through this)


def launches() -> int:
    return _launches


# ---- optional per-kernel timing (bench.py roofline): CUDA events on the launching stream around each op ----
_prof = None


def profile_start():
    global _prof
    _prof = []


def profile_stop():
    """-> [(op name, algorithmic bytes, milliseconds)] for every op issued since profile_start()."""
    global _prof
    rec, _prof = _prof or [], None
    torch.cuda.synchronize()
    return [(name, nbytes, a.elapsed_time(b)) for name, nbytes, a, b in rec]


class _P:
    __slots__ = ("name", "nbytes", "a")

    def __init__(self, name, nbytes):
        self.name, self.nbytes = name, nbytes

    def __enter__(self):
        if _prof is not None:
            self.a = torch.cuda.Event(enable_timing=True)
            self.a.record()

    def __exit__(self, *exc):
        if _prof is not None:
            b = torch.cuda.Event(enable_timing=True)
            b.record()
            _prof.append((self.name, self.nbytes, self.a, b))


def _count(n: int = 1):
    global _launches
    _launches += n


# ---- dropout seeds: host-drawn by default (reproducible under torch.manual_seed, no device sync); a provider can hand out
#      device-resident seeds instead (CUDA-graph capture, twowl_b200.graphed)
_seed_provider = None


def next_seed() -> int:
    if _seed_provider is not None:
        return _seed_provider()
    return int(torch.randint(0, 2 ** 62, (1,)).item())


def set_seed_provider(fn):
    """fn() -> int per call (or None to restore the host RNG). Returns the previous provider."""
    global _seed_provider
    prev, _seed_provider = _seed_provider, fn
    return prev


def add_launches(n: int):
    """Kernels launched outside the Python wrappers: a CUDA-graph replay of a captured step (twowl_b200.graphed)."""
    _count(int(n))


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("twowl_b200: tensors must live on a CUDA device (no CPU fallback exists)")


def _p(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _ws(nbytes: int, device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


def _row(t: torch.Tensor) -> Tuple[int, int]:
    """(data pointer, element stride) of a 1-D int64 view."""
    assert t.dim() == 1 and t.dtype == torch.int64, "expected a 1-D int64 tensor"
    return t.data_ptr(), (t.stride(0) if t.numel() > 1 else 1)


# ------------------------------------------------------------------------------ integer operators

def degree(keys: torch.Tensor, num_node: int) -> torch.Tensor:
    _need_cuda(keys)
    out = torch.empty(int(num_node), dtype=torch.int64, device=keys.device)
    p, s = _row(keys)
    check(lib.twowl_degree(p, s, keys.numel(), int(num_node), out.data_ptr(), _stream()), "degree")
    _count(2)
    return out


def csr_build(keys: torch.Tensor, num_keys: int, key_xor: int = 0, want_ptr: bool = True):
    """Stable counting sort of positions by key -> (ptr int64[num_keys+1] | None, ids int32[n])."""
    _need_cuda(keys)
    n = keys.numel()
    dev = keys.device
    ptr = torch.empty(int(num_keys) + 1, dtype=torch.int64, device=dev) if want_ptr else None
    ids = torch.empty(n, dtype=torch.int32, device=dev)
    nb = lib.twowl_csr_build_workspace_bytes(n, int(num_keys))
    ws = _ws(nb, dev)
    p, s = _row(keys)
    with _P("csr_build", n * 8 + n * 16 * 4):
        check(lib.twowl_csr_build(p, s, n, int(key_xor), int(num_keys), _p(ptr), ids.data_ptr(), ws.data_ptr(), nb,
                                  _stream()), "csr_build")
    _count(4 + 3 * 4)
    return ptr, ids


def gather_cols(ids: torch.Tensor, vals: torch.Tensor, val_xor: int = 0) -> torch.Tensor:
    _need_cuda(ids, vals)
    out = torch.empty(ids.numel(), dtype=torch.int32, device=ids.device)
    p, s = _row(vals)
    check(lib.twowl_gather_cols(ids.data_ptr(), ids.numel(), p, s, int(val_xor), out.data_ptr(), _stream()),
          "gather_cols")
    _count()
    return out


def narrow_i32(x: torch.Tensor) -> torch.Tensor:
    _need_cuda(x)
    out = torch.empty(x.numel(), dtype=torch.int32, device=x.device)
    p, s = _row(x)
    check(lib.twowl_narrow_i32(p, s, x.numel(), out.data_ptr(), _stream()), "narrow_i32")
    _count()
    return out


def ei2_offsets(in_ptr: torch.Tensor, out_ptr: torch.Tensor, n_node: int) -> torch.Tensor:
    off = torch.empty(n_node + 1, dtype=torch.int64, device=in_ptr.device)
    nb = lib.twowl_ei2_count_workspace_bytes(n_node)
    ws = _ws(nb, in_ptr.device)
    check(lib.twowl_ei2_count(in_ptr.data_ptr(), out_ptr.data_ptr(), n_node, off.data_ptr(), ws.data_ptr(), nb,
                              _stream()), "ei2_count")
    _count(4)
    return off


def ei2_fill(in_ptr, in_ids, out_ptr, out_ids, off, n_node: int, t_begin: int, t_end: int) -> torch.Tensor:
    """-> int64 [t_end - t_begin, 2] rows (a, b); its .t() is the reference's get_ei2 layout."""
    out = torch.empty((t_end - t_begin, 2), dtype=torch.int64, device=in_ptr.device)
    check(lib.twowl_ei2_fill(in_ptr.data_ptr(), in_ids.data_ptr(), out_ptr.data_ptr(), out_ids.data_ptr(),
                             off.data_ptr(), n_node, int(t_begin), int(t_end), out.data_ptr(), _stream()), "ei2_fill")
    _count()
    return out


def ei2_fill_rows(in_ptr, in_ids, out_ptr, out_ids, off, n_node: int, T: int) -> torch.Tensor:
    """-> the same wedges as a fresh contiguous int64 [2,T] tensor (rows a, b): the layout blockei2 returns."""
    out = torch.empty((2, T), dtype=torch.int64, device=in_ptr.device)
    check(lib.twowl_ei2_fill_rows(in_ptr.data_ptr(), in_ids.data_ptr(), out_ptr.data_ptr(), out_ids.data_ptr(),
                                  off.data_ptr(), n_node, 0, int(T), out.data_ptr(), _stream()), "ei2_fill_rows")
    _count()
    return out


def mask_from_idx(idx: torch.Tensor, num: int) -> torch.Tensor:
    _need_cuda(idx)
    idx = idx.reshape(-1)
    if idx.dtype != torch.int64:
        idx = idx.to(torch.int64)
    idx = idx.contiguous()
    mask = torch.empty(int(num), dtype=torch.uint8, device=idx.device)
    check(lib.twowl_mask_from_idx(idx.data_ptr(), idx.numel(), mask.data_ptr(), int(num), _stream()), "mask_from_idx")
    _count(2)
    return mask


def index_guard(idx: torch.Tensor, num: int, what: str = "index") -> torch.Tensor:
    """The bounds rule of the reference's `x[idx]` on the device, without a host sync: ids in [-num, 0) wrap, any other id
    outside [0, num) trips a device-side assertion (the way torch's own CUDA indexing reports it: the next synchronising call
    raises). Returns the wrapped ids as a contiguous int64 tensor the kernels can consume without bounds checks."""
    _need_cuda(idx)
    idx = idx.reshape(-1)
    if idx.dtype != torch.int64:
        idx = idx.to(torch.int64)
    out = torch.empty(idx.numel(), dtype=torch.int64, device=idx.device)
    bad = torch.empty(1, dtype=torch.int32, device=idx.device)
    p, s = _row(idx) if idx.numel() else (0, 1)
    check(lib.twowl_index_guard(p, s, idx.numel(), int(num), out.data_ptr(), bad.data_ptr(), _stream()), "index_guard")
    _count()
    torch._assert_async(bad == 0, f"twowl_b200: {what} out of range for {int(num)} rows (IndexError in the reference)")
    return out


def sample_non_edges(row: torch.Tensor, col: torch.Tensor, num_nodes: int, count: int, seed: Optional[int] = None,
                     undirected: bool = True, rounds: int = 16):
    """`count` distinct uniform non-edges of the graph (row[e], col[e]) on `num_nodes` nodes -> (neg_row, neg_col) int64, row < col
    when undirected (utils.py:129-146), ordered pairs otherwise (datasets.py:176-197). Deterministic under `seed` (drawn from
    torch's default generator when None, so torch.manual_seed reproduces it). Fewer than `count` pairs come back only when the
    graph does not have that many non-edges (the reference returns what exists, too) - one host read tells."""
    _need_cuda(row, col)
    row, col = row.reshape(-1), col.reshape(-1)
    assert row.dtype == torch.int64 and col.dtype == torch.int64 and row.numel() == col.numel()
    dev = row.device
    n_edges, count = row.numel(), int(count)
    out_row = torch.empty(count, dtype=torch.int64, device=dev)
    out_col = torch.empty(count, dtype=torch.int64, device=dev)
    done = torch.empty(max(count, 1), dtype=torch.uint8, device=dev)
    unresolved = torch.empty(1, dtype=torch.int32, device=dev)
    if seed is None:
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    nb = lib.twowl_nonedge_sample_workspace_bytes(n_edges, count)
    ws = _ws(nb, dev)
    (pr, sr), (pc, sc) = (_row(row), _row(col)) if n_edges else ((0, 1), (0, 1))
    check(lib.twowl_nonedge_sample(pr, sr, pc, sc, n_edges, int(num_nodes), count, int(undirected), int(seed), int(rounds),
                                   out_row.data_ptr(), out_col.data_ptr(), done.data_ptr(), unresolved.data_ptr(), ws.data_ptr(), nb,
                                   _stream()), "nonedge_sample")
    _count(1 + 2 * int(rounds))
    if count and int(unresolved.item()):        # rare: a (nearly) complete graph - keep the slots that were filled
        keep = done[:count].bool()
        out_row, out_col = out_row[keep], out_col[keep]
    return out_row, out_col


def sample_tail_negatives(row: torch.Tensor, col: torch.Tensor, num_nodes: int, src: torch.Tensor, k: int,
                          seed: Optional[int] = None, rounds: int = 16) -> torch.Tensor:
    """k distinct negatives per source for ranking evaluation -> int64 [P, k]: row i is uniform over the nodes w != src[i] such that
    neither (src[i], w) nor (w, src[i]) is an edge (row[e], col[e]) - OGB's filtered setting when the edges are every known
    positive. Deterministic under `seed` (drawn from torch's default generator when None). One host read: raises ValueError if a
    row could not be filled, i.e. a source has fewer than k allowed nodes (or is adjacent to nearly all of them: more `rounds`)."""
    _need_cuda(row, col, src)
    row, col = row.reshape(-1), col.reshape(-1)
    assert row.dtype == torch.int64 and col.dtype == torch.int64 and row.numel() == col.numel()
    src = src.reshape(-1).to(torch.int64).contiguous()
    dev = src.device
    n_edges, P, k = row.numel(), src.numel(), int(k)
    out = torch.empty((P, k), dtype=torch.int64, device=dev)
    unresolved = torch.empty(1, dtype=torch.int32, device=dev)
    if seed is None:
        seed = int(torch.randint(0, 2 ** 62, (1,)).item())
    nb = lib.twowl_tail_negative_sample_workspace_bytes(n_edges, P, k)
    ws = _ws(nb, dev)
    (pr, sr), (pc, sc) = (_row(row), _row(col)) if n_edges else ((0, 1), (0, 1))
    check(lib.twowl_tail_negative_sample(pr, sr, pc, sc, n_edges, int(num_nodes), src.data_ptr(), P, k, int(seed), int(rounds),
                                         out.data_ptr(), unresolved.data_ptr(), ws.data_ptr(), nb, _stream()), "tail_negative_sample")
    _count(1 + 2 * int(rounds))
    left = int(unresolved.item())
    if left:
        raise ValueError(f"sample_tail_negatives: {left} of {P * k} slots unfilled after {int(rounds)} rounds - a source has fewer "
                         f"than k={k} allowed nodes, lies outside [0, {int(num_nodes)}), or needs more rounds")
    return out


def select_columns(mat: torch.Tensor, mask: torch.Tensor, mode: int) -> torch.Tensor:
    """Order-preserving column selection of an int64 [2,T] matrix (any strides).
    mode 0: keep column t iff !mask[t]; mode 1: keep iff !mask[mat[0,t]]."""
    _need_cuda(mat, mask)
    assert mat.dim() == 2 and mat.shape[0] == 2 and mat.dtype == torch.int64
    T = mat.shape[1]
    dev = mat.device
    if T == 0:
        return torch.empty((2, 0), dtype=torch.int64, device=dev)
    ntiles = (T + SELECT_TILE - 1) // SELECT_TILE
    tile_off = torch.empty(ntiles + 1, dtype=torch.int64, device=dev)
    nb = lib.twowl_select_workspace_bytes(T)
    ws = _ws(nb, dev)
    (p0, s0), (p1, s1) = _row(mat[0]), _row(mat[1])
    check(lib.twowl_select_count(p0, s0, T, mask.data_ptr(), mask.numel(), mode, tile_off.data_ptr(), ws.data_ptr(), nb,
                                 _stream()), "select_count")
    t_new = int(tile_off[-1].item())  # the reference's boolean indexing synchronises here as well
    out = torch.empty((2, t_new), dtype=torch.int64, device=dev)
    check(lib.twowl_select_fill(p0, s0, p1, s1, T, mask.data_ptr(), mask.numel(), mode, tile_off.data_ptr(),
                                out[0].data_ptr() if t_new else None, out[1].data_ptr() if t_new else None, _stream()),
          "select_fill")
    _count(5)
    return out


def check_in_set(target: torch.Tensor, set_: torch.Tensor) -> torch.Tensor:
    _need_cuda(target, set_)
    target, set_ = target.reshape(-1), set_.reshape(-1).contiguous()
    n, m = target.numel(), set_.numel()
    dev = target.device
    out = torch.empty(n, dtype=torch.int64, device=dev)
    if n == 0:
        return out
    rng = int(torch.max(target.max(), set_.max() if m else target.max()).item()) + 1 if (n or m) else 1
    rng = max(rng, 1)
    counts = torch.empty(rng, dtype=torch.int32, device=dev)
    p, s = _row(target)
    check(lib.twowl_check_in_set(p, s, n, set_.data_ptr(), m, rng, counts.data_ptr(), out.data_ptr(), _stream()),
          "check_in_set")
    _count(3)
    return out


def reverse(ei2: torch.Tensor):
    _need_cuda(ei2)
    T = ei2.shape[1]
    edge = torch.empty((2, T), dtype=torch.int64, device=ei2.device)
    edge_r = torch.empty((2, T), dtype=torch.int64, device=ei2.device)
    if T:
        (p0, s0), (p1, s1) = _row(ei2[0]), _row(ei2[1])
        check(lib.twowl_reverse(p0, s0, p1, s1, T, edge.data_ptr(), edge_r.data_ptr(), _stream()), "reverse")
        _count()
    return edge, edge_r


def double_edges(x: torch.Tensor) -> torch.Tensor:
    _need_cuda(x)
    M = x.shape[1]
    out = torch.empty((2, 2 * M), dtype=torch.int64, device=x.device)
    if M:
        (p0, s0), (p1, s1) = _row(x[0]), _row(x[1])
        check(lib.twowl_double_edges(p0, s0, p1, s1, M, out.data_ptr(), _stream()), "double_edges")
        _count()
    return out


def double_index(x: torch.Tensor) -> torch.Tensor:
    _need_cuda(x)
    x = x.reshape(-1)
    out = torch.empty(2 * x.numel(), dtype=torch.int64, device=x.device)
    if x.numel():
        p, s = _row(x)
        check(lib.twowl_double_index(p, s, x.numel(), out.data_ptr(), _stream()), "double_index")
        _count()
    return out


def set_mul(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    _need_cuda(a, b)
    a, b = a.reshape(-1).contiguous(), b.reshape(-1).contiguous()
    out = torch.empty((a.numel() * b.numel(), 2), dtype=torch.int64, device=a.device)
    if out.numel():
        check(lib.twowl_set_mul(a.data_ptr(), a.numel(), b.data_ptr(), b.numel(), out.data_ptr(), _stream()), "set_mul")
        _count()
    return out


# ------------------------------------------------------------------------------ aggregation

def gcn_dinv(ptr, col, M: int, flip: int = 0, row_flip: int = 0, skip_mask=None, row_skip_mask=None) -> torch.Tensor:
    _need_cuda(ptr, col)
    dinv = torch.empty(M, dtype=torch.float32, device=ptr.device)
    check(lib.twowl_gcn_dinv(ptr.data_ptr(), col.data_ptr(), M, flip, row_flip, _p(skip_mask), _p(row_skip_mask),
                             dinv.data_ptr(), _stream()), "gcn_dinv")
    _count()
    return dinv


def gcn_dinv_entries(ptr, col, M: int, entry_mask, rows=None, out=None) -> torch.Tensor:
    """gcn_norm degree of a cached CSR minus the entries a per-entry mask removes, for the node rows rows = (lo, hi) (default: all
    M) -> out (fp32, at least M elements; a new [M] tensor by default) with out[lo:hi] written and the rest untouched."""
    _need_cuda(ptr, col, entry_mask, out)
    if out is None:
        out = torch.empty(M, dtype=torch.float32, device=ptr.device)
    assert out.dtype == torch.float32 and out.is_contiguous() and out.numel() >= M
    lo, hi = (0, M) if rows is None else rows
    check(lib.twowl_gcn_dinv_entries(ptr.data_ptr(), col.data_ptr(), M, entry_mask.data_ptr(), int(lo), int(hi), out.data_ptr(),
                                     _stream()), "gcn_dinv_entries")
    _count()
    return out


def gather_u8(mask: torch.Tensor, ids: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out[k] = mask[ids[k]] (uint8): a per-edge mask in the entry order of a CSR."""
    _need_cuda(mask, ids)
    if out is None:
        out = torch.empty(ids.numel(), dtype=torch.uint8, device=mask.device)
    assert out.dtype == torch.uint8 and out.is_contiguous() and out.numel() == ids.numel() and ids.is_contiguous()
    check(lib.twowl_gather_u8(mask.data_ptr(), ids.data_ptr(), ids.numel(), out.data_ptr(), _stream()), "gather_u8")
    _count()
    return out


LONG_ROW = 64     # TWOWL_LONG_ROW of include/twowl.h: rows with more entries go through the long-row passes of seg_reduce


def seg_plan(ptr: torch.Tensor, M: int, nnz: int) -> torch.Tensor:
    """Long-row plan of a CSR as ONE int32 tensor: [counts(2) | long_row(lc) | long_base(lc) | chunk_owner(cc)],
    lc / cc being the capacities twowl_seg_plan_{long,chunk}_cap give for nnz (no host read needed)."""
    _need_cuda(ptr)
    lc, cc = lib.twowl_seg_plan_long_cap(nnz), lib.twowl_seg_plan_chunk_cap(nnz)
    plan = torch.empty(2 + 2 * lc + cc, dtype=torch.int32, device=ptr.device)
    base = plan.data_ptr()
    check(lib.twowl_seg_plan(ptr.data_ptr(), M, nnz, base, base + 8, base + 8 + 4 * lc, base + 8 + 8 * lc, _stream()),
          "seg_plan")
    _count()
    return plan


def seg_reduce(ptr, col, M: int, X, *, plan=None, flip=0, row_flip=0, src_scale=None, skip_mask=None,
               row_skip_mask=None, skip_self=False, self_mode=0, dst_scale=None, bias=None, X2=None, mul_idx=None,
               out=None, accumulate=False, pair_sum=False, entry_mask=None, dual=False, src_scale2=None, rows=None, X_mate=None, out2=None,
               x_pairs=False):
    """dual=True -> (out, out2): out2[m] = sum src_scale2[s^1] * X[s^1] over the same entries (see twowl_seg_args).
    rows=(lo, hi): only output rows [lo, hi) are computed (and written into `out`, which keeps its full [M, C] shape)."""
    _need_cuda(ptr, col, X)
    assert X.dtype == torch.float32 and X.is_contiguous()
    C = X.shape[1]
    if out is None:
        out = torch.empty((M, C), dtype=torch.float32, device=X.device)
    if dual and out2 is None:
        out2 = torch.empty((M, C), dtype=torch.float32, device=X.device)
    a = SegArgs(ptr=ptr.data_ptr(), col=col.data_ptr(), M=M, X=X.data_ptr(), C=C, flip=int(flip), row_flip=int(row_flip),
                src_scale=_p(src_scale), skip_mask=_p(skip_mask), row_skip_mask=_p(row_skip_mask),
                skip_self=int(skip_self), self_mode=int(self_mode), dst_scale=_p(dst_scale), bias=_p(bias), X2=_p(X2),
                mul_idx=_p(mul_idx), out=out.data_ptr(), accumulate=int(accumulate), pair_sum=2 if x_pairs else int(pair_sum),
                entry_mask=_p(entry_mask))
    if rows is not None:
        a.row_begin, a.row_end = int(rows[0]), int(rows[1])
        if a.row_end <= a.row_begin:
            return (out, out2) if dual else out
    partial = None
    if plan is not None:
        nnz = col.numel()
        lc, cc = lib.twowl_seg_plan_long_cap(nnz), lib.twowl_seg_plan_chunk_cap(nnz)
        assert plan.numel() == 2 + 2 * lc + cc, "plan does not belong to this CSR"
        partial = torch.empty((cc, C), dtype=torch.float32, device=X.device)
        base = plan.data_ptr()
        a.plan_counts, a.long_row, a.long_base, a.chunk_owner = base, base + 8, base + 8 + 4 * lc, base + 8 + 8 * lc
        a.partial, a.chunk_cap, a.long_cap = partial.data_ptr(), cc, lc
        if dual:
            partial2 = torch.empty((cc, C), dtype=torch.float32, device=X.device)
            a.partial2 = partial2.data_ptr()
    if dual:
        a.src_scale2, a.out2 = _p(src_scale2), out2.data_ptr()
        if X_mate is not None:      # the mates' rows come from a second matrix of the same shape (dO_r next to dO_f)
            assert X_mate.shape == X.shape and X_mate.is_contiguous() and X_mate.dtype == torch.float32
            a.X_mate = X_mate.data_ptr()
    nbytes = col.numel() * (4 * C * (1 + int(pair_sum) + int(X2 is not None) + int(dual and not x_pairs)) + 8 + 4 * int(dual)) + \
        M * (4 * C + 8) * (1 + int(dual))
    if rows is not None:      # a node block: its share of the entries is not known on the host - charged by its share of the rows
        nbytes = nbytes * (int(rows[1]) - int(rows[0])) // max(M, 1)
    with _P("seg_reduce", nbytes):
        check(lib.twowl_seg_reduce(ctypes.byref(a), _stream()), "seg_reduce")
    _count(1 if plan is None else 3)
    return (out, out2) if dual else out


def gather_rows(W: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    _need_cuda(W, idx)
    idx = idx.reshape(-1)
    out = torch.empty((idx.numel(), W.shape[1]), dtype=torch.float32, device=W.device)
    p, s = _row(idx)
    with _P("gather_rows", idx.numel() * (8 * W.shape[1] + 8)):
        check(lib.twowl_gather_rows(W.data_ptr(), W.shape[0], p, s, idx.numel(), W.shape[1], out.data_ptr(), _stream()),
              "gather_rows")
    _count()
    return out


def pair_init_fwd(X, src32, dst32, pairs: bool = False) -> torch.Tensor:
    """H[p] = X[src[p]] * X[dst[p]]; pairs=True on a mated table: ONE row per pair, H[k] = X[src[2k]] * X[dst[2k]] ([R/2, C])."""
    _need_cuda(X, src32, dst32)
    R = src32.numel()
    rows = R // 2 if pairs else R
    out = torch.empty((rows, X.shape[1]), dtype=torch.float32, device=X.device)
    with _P("pair_init_fwd", rows * (12 * X.shape[1] + 8)):
        check(lib.twowl_pair_init_fwd(X.data_ptr(), src32.data_ptr(), dst32.data_ptr(), R, X.shape[1], int(pairs), out.data_ptr(),
                                      _stream()), "pair_init_fwd")
    _count()
    return out


def readout_fwd(H, idx, w, b) -> torch.Tensor:
    _need_cuda(H, idx, w, b)
    idx = idx.reshape(-1)
    L = idx.numel() // 2
    pred = torch.empty((L, 1), dtype=torch.float32, device=H.device)
    p, s = _row(idx)
    with _P("readout_fwd", L * (8 * H.shape[1] + 20)):
        check(lib.twowl_readout_fwd(H.data_ptr(), p, s, L, H.shape[1], w.data_ptr(), b.data_ptr(), pred.data_ptr(),
                                    _stream()), "readout_fwd")
    _count()
    return pred


def readout_bwd(H, idx, w, dpred):
    idx = idx.reshape(-1)
    L = idx.numel() // 2
    C = H.shape[1]
    dev = H.device
    _, order = csr_build(idx[: 2 * L], H.shape[0], want_ptr=False)
    dH = torch.zeros_like(H)
    dw = torch.empty((1, C), dtype=torch.float32, device=dev)
    db = torch.empty(1, dtype=torch.float32, device=dev)
    nb = lib.twowl_readout_bwd_workspace_bytes(L, C)
    ws = _ws(nb, dev)
    p, s = _row(idx)
    dpred = dpred.contiguous()
    with _P("readout_bwd", H.numel() * 4 + L * (28 * C + 24)):
        check(lib.twowl_readout_bwd(H.data_ptr(), p, s, L, C, w.data_ptr(), dpred.data_ptr(), order.data_ptr(),
                                    dH.data_ptr(), dw.data_ptr(), db.data_ptr(), ws.data_ptr(), nb, _stream()), "readout_bwd")
    _count(6)
    return dH, dw, db


def gn2_readout_fwd(xf, xr, sf, sr, pf, pr, p_drop: float, seed_f: int, seed_r: int, relu: bool, idx, w, b) -> torch.Tensor:
    """pred[l] of model.py:78-83 straight from the two pre-GraphNorm branch outputs (last pair layer): only the rows
    idx selects are normalised / activated. pf / pr = (weight, bias, mean_scale) of the two GraphNorms."""
    _need_cuda(xf, xr, idx, w, b)
    M, C = xf.shape
    idx = idx.reshape(-1)
    L = idx.numel() // 2
    pred = torch.empty((L, 1), dtype=torch.float32, device=xf.device)
    p, s = _row(idx)
    with _P("gn2_readout_fwd", L * (16 * C + 20)):
        check(lib.twowl_gn2_readout_fwd(xf.data_ptr(), xr.data_ptr(), M, C, sf.data_ptr(), sr.data_ptr(), pf[0].data_ptr(),
                                        pf[1].data_ptr(), pf[2].data_ptr(), pr[0].data_ptr(), pr[1].data_ptr(), pr[2].data_ptr(),
                                        float(p_drop), int(seed_f), int(seed_r), int(relu), p, s, L, w.data_ptr(), b.data_ptr(),
                                        pred.data_ptr(), _stream()), "gn2_readout_fwd")
    _count()
    return pred


def gn2_readout_bwd(xf, xr, sf, sr, pf, pr, p_drop: float, seed_f: int, seed_r: int, relu: bool, idx, w, dpred):
    """-> (dxf, dxr [M,C], dparams_f, dparams_r [4C], dw [1,C], db [1]) from dpred [L]."""
    M, C = xf.shape
    dev = xf.device
    idx = idx.reshape(-1)
    L = idx.numel() // 2
    dxf, dxr = torch.empty_like(xf), torch.empty_like(xr)
    dpf = torch.empty(4 * C, dtype=torch.float32, device=dev)
    dpr = torch.empty(4 * C, dtype=torch.float32, device=dev)
    dw = torch.empty((1, C), dtype=torch.float32, device=dev)
    db = torch.empty(1, dtype=torch.float32, device=dev)
    nb = lib.twowl_gn2_readout_bwd_workspace_bytes(M, L, C)
    ws = _ws(nb, dev)
    p, s = _row(idx)
    dpred = dpred.contiguous()
    with _P("gn2_readout_bwd", M * (16 * C + 4) + L * (48 * C + 40)):
        check(lib.twowl_gn2_readout_bwd(xf.data_ptr(), xr.data_ptr(), M, C, sf.data_ptr(), sr.data_ptr(), pf[0].data_ptr(),
                                        pf[1].data_ptr(), pf[2].data_ptr(), pr[0].data_ptr(), pr[1].data_ptr(), pr[2].data_ptr(),
                                        float(p_drop), int(seed_f), int(seed_r), int(relu), p, s, L, w.data_ptr(), dpred.data_ptr(),
                                        dxf.data_ptr(), dxr.data_ptr(), dpf.data_ptr(), dpr.data_ptr(), dw.data_ptr(), db.data_ptr(),
                                        ws.data_ptr(), nb, _stream()), "gn2_readout_bwd")
    _count(8)
    return dxf, dxr, dpf, dpr, dw, db


def gn2_readout_bwd_prepare(xf, xr, sf, sr, pf, pr, p_drop: float, seed_f: int, seed_r: int, relu: bool, idx, w, dpred,
                            M_total: Optional[int] = None, all_reduce=None):
    """The row-sparse part of gn2_readout_bwd for a consumer that makes dxf / dxr on the fly (pair_dw_gn):
    -> (G [2L,C], head int32[M], next int32[2L], consts [8C], dparams_f, dparams_r [4C], dw [1,C], db [1]).
    On one row block of a row-sharded pair table, `all_reduce` (a callable applied in place) sums the fp64 column sums [6,C] over
    the ranks between the two halves, and M_total is the whole table's row count (default: M)."""
    M, C = xf.shape
    dev = xf.device
    idx = idx.reshape(-1)
    L = idx.numel() // 2
    G = torch.empty((max(2 * L, 1), C), dtype=torch.float32, device=dev)
    head = torch.empty(M, dtype=torch.int32, device=dev)
    nxt = torch.empty(max(2 * L, 1), dtype=torch.int32, device=dev)
    colsums = torch.empty((6, C), dtype=torch.float64, device=dev)
    nb = lib.twowl_gn2_readout_bwd_rows_workspace_bytes(M, L, C)
    ws = _ws(nb, dev)
    p, s = _row(idx) if L > 0 else (0, 1)
    dpred = dpred.contiguous()
    with _P("gn2_readout_bwd_prepare", M * 4 + L * (48 * C + 40)):
        check(lib.twowl_gn2_readout_bwd_rows(xf.data_ptr(), xr.data_ptr(), M, C, sf.data_ptr(), sr.data_ptr(), pf[0].data_ptr(),
                                             pf[1].data_ptr(), pf[2].data_ptr(), pr[0].data_ptr(), pr[1].data_ptr(),
                                             pr[2].data_ptr(), float(p_drop), int(seed_f), int(seed_r), int(relu), p, s, L,
                                             w.data_ptr(), dpred.data_ptr(), G.data_ptr(), head.data_ptr(), nxt.data_ptr(),
                                             colsums.data_ptr(), ws.data_ptr(), nb, _stream()), "gn2_readout_bwd_rows")
    _count(4)
    if all_reduce is not None:
        all_reduce(colsums)
    consts = torch.empty(8 * C, dtype=torch.float32, device=dev)
    dpf = torch.empty(4 * C, dtype=torch.float32, device=dev)
    dpr = torch.empty(4 * C, dtype=torch.float32, device=dev)
    dw = torch.empty((1, C), dtype=torch.float32, device=dev)
    db = torch.empty(1, dtype=torch.float32, device=dev)
    nb = lib.twowl_gn2_readout_bwd_finish_workspace_bytes(C)
    ws = _ws(nb, dev)
    check(lib.twowl_gn2_readout_bwd_finish(colsums.data_ptr(), int(M if M_total is None else M_total), C, sf.data_ptr(), sr.data_ptr(),
                                           pf[0].data_ptr(), pf[1].data_ptr(), pf[2].data_ptr(), pr[0].data_ptr(), pr[1].data_ptr(),
                                           pr[2].data_ptr(), consts.data_ptr(), dpf.data_ptr(), dpr.data_ptr(), dw.data_ptr(),
                                           db.data_ptr(), ws.data_ptr(), nb, _stream()), "gn2_readout_bwd_finish")
    _count(6)
    return G, head, nxt, consts, dpf, dpr, dw, db


# ------------------------------------------------------------------------------ GraphNorm

def graphnorm_stats_from_moments(moments, M_total: int, mean_scale, eps: float) -> torch.Tensor:
    """GraphNorm (mean, inv_std)[2C] from the rank-summed column (sum, sum of squares) float64[2C] over M_total rows."""
    _need_cuda(moments, mean_scale)
    C = mean_scale.numel()
    stats = torch.empty(2 * C, dtype=torch.float32, device=moments.device)
    check(lib.twowl_graphnorm_stats_from_moments(moments.data_ptr(), int(M_total), C, mean_scale.data_ptr(), float(eps),
                                                 stats.data_ptr(), _stream()), "graphnorm_stats_from_moments")
    _count()
    return stats


def graphnorm_stats(x, mean_scale, eps: float) -> torch.Tensor:
    _need_cuda(x)
    M, C = x.shape
    stats = torch.empty(2 * C, dtype=torch.float32, device=x.device)
    nb = lib.twowl_graphnorm_stats_workspace_bytes(M, C)
    ws = _ws(nb, x.device)
    with _P("graphnorm_stats", M * C * 4):
        check(lib.twowl_graphnorm_stats(x.data_ptr(), M, C, mean_scale.data_ptr(), float(eps), stats.data_ptr(),
                                        ws.data_ptr(), nb, _stream()), "graphnorm_stats")
    _count(2)
    return stats


def graphnorm_apply(x, stats, weight, bias, mean_scale, p_drop: float, seed: int, relu: bool, addend=None):
    M, C = x.shape
    out = torch.empty_like(x)
    with _P("graphnorm_apply", M * C * 4 * (2 if addend is None else 3)):
        check(lib.twowl_graphnorm_apply(x.data_ptr(), M, C, stats.data_ptr(), weight.data_ptr(), bias.data_ptr(),
                                        mean_scale.data_ptr(), float(p_drop), int(seed), int(relu), _p(addend),
                                        out.data_ptr(), _stream()), "graphnorm_apply")
    _count()
    return out


def graphnorm_bwd(x, dout, stats, weight, bias, mean_scale, p_drop: float, seed: int, relu: bool):
    M, C = x.shape
    dx = torch.empty_like(x)
    dparams = torch.empty(4 * C, dtype=torch.float32, device=x.device)
    nb = lib.twowl_graphnorm_bwd_workspace_bytes(M, C)
    ws = _ws(nb, x.device)
    with _P("graphnorm_bwd", M * C * 4 * 5):
        check(lib.twowl_graphnorm_bwd(x.data_ptr(), dout.data_ptr(), M, C, stats.data_ptr(), weight.data_ptr(),
                                      bias.data_ptr(), mean_scale.data_ptr(), float(p_drop), int(seed), int(relu),
                                      dx.data_ptr(), dparams.data_ptr(), ws.data_ptr(), nb, _stream()), "graphnorm_bwd")
    _count(3)
    return dx, dparams


def colsum(x) -> torch.Tensor:
    M, C = x.shape
    out = torch.empty(C, dtype=torch.float32, device=x.device)
    nb = lib.twowl_colsum_workspace_bytes(M, C)
    ws = _ws(nb, x.device)
    with _P("colsum", M * C * 4):
        check(lib.twowl_colsum(x.data_ptr(), M, C, out.data_ptr(), ws.data_ptr(), nb, _stream()), "colsum")
    _count(2)
    return out


# ------------------------------------------------------------------------------ linear

# 0 = SIMT FFMA (exact fp32), 1 = tcgen05 3xTF32 (error when the shape is unsupported), 2 = tcgen05 where supported
LINEAR_IMPL = int(os.environ.get("TWOWL_LINEAR_IMPL", "2"))


def linear_fwd(X, W, impl: int = -1) -> torch.Tensor:
    _need_cuda(X, W)
    M, Ci = X.shape
    Co = W.shape[0]
    Z = torch.empty((M, Co), dtype=torch.float32, device=X.device)
    impl = LINEAR_IMPL if impl < 0 else impl
    with _P("linear_fwd", 4 * M * (Ci + Co)):
        check(lib.twowl_linear_fwd(X.data_ptr(), W.data_ptr(), M, Ci, Co, Z.data_ptr(), impl, _stream()), "linear_fwd")
    _count()
    return Z


def linear_bwd_input(dZ, W, impl: int = -1) -> torch.Tensor:
    M, Co = dZ.shape
    Ci = W.shape[1]
    dX = torch.empty((M, Ci), dtype=torch.float32, device=dZ.device)
    impl = LINEAR_IMPL if impl < 0 else impl
    with _P("linear_bwd_input", 4 * M * (Ci + Co)):
        check(lib.twowl_linear_bwd_input(dZ.data_ptr(), W.data_ptr(), M, Ci, Co, dX.data_ptr(), impl, _stream()),
              "linear_bwd_input")
    _count()
    return dX


def linear_bwd_weight(dZ, X, row_scale=None) -> torch.Tensor:
    M, Co = dZ.shape
    Ci = X.shape[1]
    dW = torch.empty((Co, Ci), dtype=torch.float32, device=dZ.device)
    nb = lib.twowl_linear_bwd_weight_workspace_bytes(M, Ci, Co)
    ws = _ws(nb, dZ.device)
    with _P("linear_bwd_weight", 4 * M * (Ci + Co)):
        check(lib.twowl_linear_bwd_weight_scaled(dZ.data_ptr(), _p(row_scale), X.data_ptr(), M, Ci, Co, dW.data_ptr(),
                                                 ws.data_ptr(), nb, _stream()), "linear_bwd_weight")
    _count(2)
    return dW


# ------------------------------------------------------------------------------ node-attribute input (model.py:47-51)

def dropout(x, p: float, seed: int) -> torch.Tensor:
    """nn.Dropout(p) with the mask a counter hash of (seed, flat index): the same call on a gradient is the backward."""
    _need_cuda(x)
    x = x.contiguous()
    out = torch.empty_like(x)
    check(lib.twowl_dropout(x.data_ptr(), x.numel(), float(p), int(seed), out.data_ptr(), _stream()), "dropout")
    _count()
    return out


def bias_layernorm_fwd(z, bias, eps: float, p_drop: float, seed: int):
    """dropout(LayerNorm(z + bias)) without affine parameters -> (y [M,C], stats [M,2] = (mean, inv_std))."""
    _need_cuda(z, bias)
    M, C = z.shape
    y = torch.empty_like(z)
    stats = torch.empty((M, 2), dtype=torch.float32, device=z.device)
    with _P("bias_layernorm_fwd", 8 * M * C):
        check(lib.twowl_bias_layernorm_fwd(z.data_ptr(), _p(bias), M, C, float(eps), float(p_drop), int(seed), y.data_ptr(),
                                           stats.data_ptr(), _stream()), "bias_layernorm_fwd")
    _count()
    return y, stats


def bias_layernorm_bwd(g, z, bias, stats, p_drop: float, seed: int) -> torch.Tensor:
    M, C = z.shape
    dz = torch.empty_like(z)
    with _P("bias_layernorm_bwd", 12 * M * C):
        check(lib.twowl_bias_layernorm_bwd(g.data_ptr(), z.data_ptr(), _p(bias), stats.data_ptr(), M, C, float(p_drop), int(seed),
                                           dz.data_ptr(), _stream()), "bias_layernorm_bwd")
    _count()
    return dz


# ------------------------------------------------------------------------------ structured wedge path

def wedge_prepare(src32, dst_e32, E: int, R: int, N: int, blocked, in_ptr, ranges=None):
    """Per-row constants of the pair rows ranges = ((lo0, hi0), (lo1, hi1)), written one range after the other (default: the whole
    table, ((0, R), (R, R))) -> (cnt [N], centre, dinv, selfw, bnode [2, (hi0 - lo0) + (hi1 - lo1)])."""
    (lo0, hi0), (lo1, hi1) = ((0, R), (R, R)) if ranges is None else ranges
    dev = src32.device
    Rl = (hi0 - lo0) + (hi1 - lo1)
    cnt = torch.empty(max(N, 1), dtype=torch.int32, device=dev)
    centre = torch.empty((2, Rl), dtype=torch.int32, device=dev)
    dinv = torch.empty((2, Rl), dtype=torch.float32, device=dev)
    selfw = torch.empty((2, Rl), dtype=torch.float32, device=dev)
    bnode = torch.empty((2, Rl), dtype=torch.int32, device=dev)
    check(lib.twowl_wedge_prepare(src32.data_ptr(), dst_e32.data_ptr(), E, R, N, _p(blocked), in_ptr.data_ptr(), int(lo0), int(hi0),
                                  int(lo1), int(hi1), cnt.data_ptr(), centre.data_ptr(), dinv.data_ptr(), selfw.data_ptr(),
                                  bnode.data_ptr(), _stream()), "wedge_prepare")
    _count(2 + (hi0 > lo0) + (hi1 > lo1))
    return cnt, centre, dinv, selfw, bnode


def wedge_apply_fwd(S, Z, centre, dinv, selfw, bias) -> torch.Tensor:
    R, C = Z.shape
    out = torch.empty_like(Z)
    with _P("wedge_apply_fwd", R * (12 * C + 12)):
        check(lib.twowl_wedge_apply_fwd(S.data_ptr(), Z.data_ptr(), centre.data_ptr(), dinv.data_ptr(), selfw.data_ptr(),
                                        _p(bias), R, C, out.data_ptr(), _stream()), "wedge_apply_fwd")
    _count()
    return out


def wedge_apply_bwd(dS, dO, dst_e32, blocked, E: int, N: int, dinv, selfw, direction: int) -> torch.Tensor:
    R, C = dO.shape
    dZ = torch.empty_like(dO)
    with _P("wedge_apply_bwd", R * (12 * C + 12)):
        check(lib.twowl_wedge_apply_bwd(dS.data_ptr(), dO.data_ptr(), dst_e32.data_ptr(), _p(blocked), E, N,
                                        dinv.data_ptr(), selfw.data_ptr(), direction, R, C, dZ.data_ptr(), _stream()),
              "wedge_apply_bwd")
    _count()
    return dZ


# ------------------------------------------------------------------------------ fused tensor-core pair layer

def pair_conv_supported(Kd: int, Nd: int, nsrc: int) -> bool:
    return bool(lib.twowl_pair_conv_supported(Kd, Nd, nsrc))


def pair_conv(A, W, w_kn, *, row_scale=None, gathers=(), bias=None, stats_mean_scale=None, eps: float = 1e-5,
              want_moments: bool = False, out=None, pair_sum_out: bool = False, a_pairs: bool = False):
    """out = sum_s (row_scale_s * A_s) B_s^T + sum_g coef_g * T_g[idx_g] + bias on tcgen05 (3xTF32).
    A, W, w_kn, row_scale: sequences of length nsrc; gathers: sequence of (T, idx int32, coef).
    Returns out, or (out, stats[2*Nd]) when stats_mean_scale is given (GraphNorm mean / inv_std of out), or
    (out, moments float64[2*Nd]) with want_moments (raw column sum / sum of squares, for a row-sharded caller).
    pair_sum_out: out is [M/2, Nd] and holds out[2k] + out[2k+1] (what the pair-init backward consumes: seg_reduce(x_pairs=True)).
    a_pairs: A[0] holds ONE row per pair ([M/2, Kd], pair_init_fwd(pairs=True)) and output row r uses row r >> 1; out keeps M rows."""
    nsrc = len(A)
    M, Kd = A[0].shape
    if a_pairs:
        M *= 2
    Nd = W[0].shape[1] if w_kn[0] else W[0].shape[0]
    dev = A[0].device
    _need_cuda(*A, *W)
    Mo = M // 2 if pair_sum_out else M
    if pair_sum_out:
        assert M % 2 == 0 and stats_mean_scale is None, "pair_conv: pair_sum_out needs an even M and no statistics"
    if out is None:
        out = torch.empty((Mo, Nd), dtype=torch.float32, device=dev)
    else:   # a caller-owned [M, Nd] buffer that is none of this launch's inputs (the in-place backward, see INPLACE_BACKWARD)
        assert out.shape == (Mo, Nd) and out.is_contiguous() and all(out.data_ptr() != x.data_ptr() for x in A)
    a = ConvArgs(nsrc=nsrc, ngather=len(gathers), Kd=Kd, Nd=Nd, M=M, bias=_p(bias), out=out.data_ptr(), eps=float(eps),
                 pair_sum_out=int(pair_sum_out), a_pairs=int(a_pairs))
    keep = []
    for s in range(nsrc):
        x = A[s].contiguous()
        keep.append(x)
        a.A[s], a.W[s], a.w_kn[s] = x.data_ptr(), W[s].data_ptr(), int(w_kn[s])
        a.row_scale[s] = _p(row_scale[s]) if row_scale is not None else None
    for g, (T, idx, coef) in enumerate(gathers):
        a.T[g], a.tidx[g], a.tcoef[g] = T.data_ptr(), idx.data_ptr(), coef.data_ptr()
    stats, ws, nb = None, None, 0
    if stats_mean_scale is not None:
        stats = torch.empty(2 * Nd, dtype=torch.float32, device=dev)
        nb = lib.twowl_pair_conv_workspace_bytes(M, Nd)
        ws = _ws(nb, dev)
        a.stats, a.mean_scale = stats.data_ptr(), stats_mean_scale.data_ptr()
    moments = None
    if want_moments:
        assert stats is not None, "pair_conv: moments need stats_mean_scale"
        moments = torch.zeros(2 * Nd, dtype=torch.float64, device=dev)   # zeros: an empty row block contributes nothing
        a.moments = moments.data_ptr()
    nbytes = (M // 2 if a_pairs else M) * 4 * Kd * nsrc + M * (8 * len(gathers) + (4 * Nd + 8) * len(gathers)) + Mo * 4 * Nd
    with _P("pair_conv", nbytes):
        check(lib.twowl_pair_conv(ctypes.byref(a), _p(ws), nb, _stream()), "pair_conv")
    _count(1 if stats is None else 2)
    if moments is not None:
        return out, moments
    return out if stats is None else (out, stats)


def pair_dw_supported(C: int) -> bool:
    return bool(lib.twowl_pair_dw_supported(C))


def pair_dw(dOf, dOr, rsf, rsr, H):
    """(dWf, dWr) = ((rsf*dOf)^T H, (rsr*dOr)^T H) in one pass on tcgen05 (3xTF32)."""
    _need_cuda(dOf, dOr, H)
    M, C = H.shape
    dWf = torch.empty((C, C), dtype=torch.float32, device=H.device)
    dWr = torch.empty((C, C), dtype=torch.float32, device=H.device)
    nb = lib.twowl_pair_dw_workspace_bytes(M, C)
    ws = _ws(nb, H.device)
    with _P("pair_dw", 12 * M * C + 8 * M):
        check(lib.twowl_pair_dw(dOf.data_ptr(), dOr.data_ptr(), rsf.data_ptr(), rsr.data_ptr(), H.data_ptr(), M, C,
                                dWf.data_ptr(), dWr.data_ptr(), ws.data_ptr(), nb, _stream()), "pair_dw")
    _count(2)
    return dWf, dWr


def pair_dw_wide_supported(Co: int, Ci: int) -> bool:
    """Widths beyond the single-launch kernel, tiled into 128-column blocks."""
    return Co > 128 and Co % 128 == 0 and Ci % 128 == 0 and Co <= 1024 and Ci <= 1024


def pair_dw_wide(dOf, dOr, rsf, rsr, H):
    """pair_dw for layers wider than 128: one tcgen05 launch per (128-column block of dO, 128-column block of H) through TMA
    tensor maps with a row pitch (twowl_pair_dw_ld) -> (dWf, dWr) [Co, Ci]."""
    _need_cuda(dOf, dOr, H)
    M, Co = dOf.shape
    Ci = H.shape[1]
    B = 128
    dWf = torch.empty((Co, Ci), dtype=torch.float32, device=H.device)
    dWr = torch.empty((Co, Ci), dtype=torch.float32, device=H.device)
    nb = lib.twowl_pair_dw_workspace_bytes(M, B)
    ws = _ws(nb, H.device)
    tf = torch.empty((B, B), dtype=torch.float32, device=H.device)
    tr = torch.empty((B, B), dtype=torch.float32, device=H.device)
    for i in range(Co // B):
        for j in range(Ci // B):
            with _P("pair_dw", 12 * M * B + 8 * M):
                check(lib.twowl_pair_dw_ld(dOf.data_ptr() + 4 * i * B, dOr.data_ptr() + 4 * i * B, rsf.data_ptr(), rsr.data_ptr(),
                                           H.data_ptr() + 4 * j * B, M, B, Co, Ci, tf.data_ptr(), tr.data_ptr(), ws.data_ptr(), nb,
                                           _stream()), "pair_dw_ld")
            _count(2)
            dWf[i * B:(i + 1) * B, j * B:(j + 1) * B] = tf
            dWr[i * B:(i + 1) * B, j * B:(j + 1) * B] = tr
    return dWf, dWr


# The backward of the last pair layer may reuse the forward's buffers: dO_f / dO_r are written over O_f / O_r (every 64-row
# tile is read by the CTA that overwrites it) and dH over H (which that launch does not read). 3 live [R,C] tensors instead of 6:
# hidden 128 at R = 60 M pair rows fits one 180 GB GPU. The saved activations are gone afterwards, so backward(retain_graph=True)
# is not possible in this mode - opt in with TWOWL_INPLACE_BACKWARD=1 or ops.INPLACE_BACKWARD = True.
INPLACE_BACKWARD = os.environ.get("TWOWL_INPLACE_BACKWARD", "0") != "0"


def pair_dw_gn(Of, Or, consts, G, head, nxt, p_drop: float, seed_f: int, seed_r: int, relu: bool, rsf, rsr, H, inplace: bool = False):
    """pair_dw with the gradients made on the fly from the last pair layer's outputs (after gn2_readout_bwd_prepare):
    -> (dOf, dOr [M,C], dWf, dWr [C,C]). One pass: reads Of, Or, H, writes dOf, dOr (over Of, Or with inplace=True).
    H may hold ONE row per pair ([M/2, C], pair_init_fwd(pairs=True)): it then stands for rows 2k and 2k+1."""
    _need_cuda(Of, Or, H)
    M, C = Of.shape
    h_pairs = H.shape[0] != M
    assert H.shape == ((M // 2, C) if h_pairs else (M, C)) and (M % 2 == 0 or not h_pairs), "pair_dw_gn: H is [M, C] or [M/2, C]"
    dOf, dOr = (Of, Or) if inplace else (torch.empty_like(Of), torch.empty_like(Or))
    dWf = torch.empty((C, C), dtype=torch.float32, device=H.device)
    dWr = torch.empty((C, C), dtype=torch.float32, device=H.device)
    nb = lib.twowl_pair_dw_workspace_bytes(M, C)
    ws = _ws(nb, H.device)
    with _P("pair_dw_gn", (18 if h_pairs else 20) * M * C + 12 * M):
        check(lib.twowl_pair_dw_gn(Of.data_ptr(), Or.data_ptr(), consts.data_ptr(), G.data_ptr(), head.data_ptr(), nxt.data_ptr(),
                                   float(p_drop), int(seed_f), int(seed_r), int(relu), rsf.data_ptr(), rsr.data_ptr(), H.data_ptr(),
                                   int(h_pairs), M, C, dOf.data_ptr(), dOr.data_ptr(), dWf.data_ptr(), dWr.data_ptr(), ws.data_ptr(), nb,
                                   _stream()), "pair_dw_gn")
    _count(2)
    return dOf, dOr, dWf, dWr


def graphnorm_apply2(xf, xr, sf, sr, pf, pr, p_drop: float, seed_f: int, seed_r: int, relu: bool):
    """pf / pr = (weight, bias, mean_scale) of the two GraphNorms."""
    M, C = xf.shape
    out = torch.empty_like(xf)
    with _P("graphnorm_apply2", M * C * 4 * 3):
        check(lib.twowl_graphnorm_apply2(xf.data_ptr(), xr.data_ptr(), M, C, sf.data_ptr(), sr.data_ptr(), pf[0].data_ptr(),
                                         pf[1].data_ptr(), pf[2].data_ptr(), pr[0].data_ptr(), pr[1].data_ptr(),
                                         pr[2].data_ptr(), float(p_drop), int(seed_f), int(seed_r), int(relu), out.data_ptr(),
                                         _stream()), "graphnorm_apply2")
    _count()
    return out


def graphnorm_bwd2(xf, xr, dout, sf, sr, pf, pr, p_drop: float, seed_f: int, seed_r: int, relu: bool, M_total: Optional[int] = None,
                   all_reduce=None):
    """Backward of graphnorm_apply2 -> (dxf, dxr, dparams_f, dparams_r). On one row block of a row-sharded pair table,
    `all_reduce` (a callable applied in place) sums the fp64 column sums [4,C] over the ranks between the two halves, and M_total
    is the whole table's row count (default: M)."""
    M, C = xf.shape
    dev = xf.device
    colsums = torch.empty((4, C), dtype=torch.float64, device=dev)
    nb = lib.twowl_graphnorm_bwd2_sums_workspace_bytes(M, C)
    ws = _ws(nb, dev)
    ptrs = (sf.data_ptr(), sr.data_ptr(), pf[0].data_ptr(), pf[1].data_ptr(), pf[2].data_ptr(), pr[0].data_ptr(), pr[1].data_ptr(),
            pr[2].data_ptr(), float(p_drop), int(seed_f), int(seed_r), int(relu))
    with _P("graphnorm_bwd2", M * C * 4 * 3):
        check(lib.twowl_graphnorm_bwd2_sums(xf.data_ptr(), xr.data_ptr(), dout.data_ptr(), M, C, *ptrs, colsums.data_ptr(),
                                            ws.data_ptr(), nb, _stream()), "graphnorm_bwd2_sums")
    _count(2)
    if all_reduce is not None:
        all_reduce(colsums)
    dxf, dxr = torch.empty_like(xf), torch.empty_like(xr)
    dpf = torch.empty(4 * C, dtype=torch.float32, device=dev)
    dpr = torch.empty(4 * C, dtype=torch.float32, device=dev)
    nb2 = lib.twowl_graphnorm_bwd2_apply_workspace_bytes(C)
    ws2 = _ws(nb2, dev)
    with _P("graphnorm_bwd2", M * C * 4 * 5):
        check(lib.twowl_graphnorm_bwd2_apply(xf.data_ptr(), xr.data_ptr(), dout.data_ptr(), M, C, *ptrs, colsums.data_ptr(),
                                             int(M if M_total is None else M_total), dxf.data_ptr(), dxr.data_ptr(), dpf.data_ptr(),
                                             dpr.data_ptr(), ws2.data_ptr(), nb2, _stream()), "graphnorm_bwd2_apply")
    _count(3)
    return dxf, dxr, dpf, dpr


# ------------------------------------------------------------------------------ loss + optimiser (train.py:37-39)

def bce_logits(logits: torch.Tensor, labels: torch.Tensor, want_grad: bool = True, want_prob: bool = False):
    """F.binary_cross_entropy_with_logits (mean) forward and backward in one pass -> (loss [1], dlogits like logits | None,
    sigmoid(logits) | None)."""
    _need_cuda(logits, labels)
    x = logits.detach().reshape(-1).contiguous()
    y = labels.detach().reshape(-1).to(torch.float32).contiguous()
    n = x.numel()
    assert y.numel() == n and x.dtype == torch.float32, "bce_logits: fp32 logits and as many labels"
    dev = x.device
    loss = torch.empty(1, dtype=torch.float32, device=dev)
    dx = torch.empty_like(x) if want_grad else None
    prob = torch.empty_like(x) if want_prob else None
    nb = lib.twowl_bce_logits_workspace_bytes(n)
    ws = _ws(nb, dev)
    check(lib.twowl_bce_logits(x.data_ptr(), y.data_ptr(), n, loss.data_ptr(), _p(dx), _p(prob), ws.data_ptr(), nb, _stream()), "bce_logits")
    _count(2)
    return loss, (None if dx is None else dx.view_as(logits)), (None if prob is None else prob.view_as(logits))


def adam_step(param, grad, exp_avg, exp_avg_sq, step, lr: float, beta1: float, beta2: float, eps: float, weight_decay: float = 0.0,
              grad_scale=None):
    """torch.optim.Adam.step() over one flat fp32 buffer, in place; `step` = int64 device scalar (incremented)."""
    _need_cuda(param, grad, exp_avg, exp_avg_sq, step)
    n = param.numel()
    assert grad.numel() == n and exp_avg.numel() == n and exp_avg_sq.numel() == n and step.dtype == torch.int64
    assert all(t.is_contiguous() and t.dtype == torch.float32 for t in (param, grad, exp_avg, exp_avg_sq))
    check(lib.twowl_adam_step(param.data_ptr(), grad.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(), n, float(lr), float(beta1),
                              float(beta2), float(eps), float(weight_decay), _p(grad_scale), step.data_ptr(), _stream()), "adam_step")
    _count(2)


# ------------------------------------------------------------------------------ metrics

def auc(score: torch.Tensor, label: torch.Tensor) -> torch.Tensor:
    """ROC-AUC of fp32 scores against {0,1} labels on the device -> float64[3] = (auc, n_pos, n_neg), no host sync.
    Ties share their average rank, as sklearn.metrics.roc_auc_score (train.py:41-43, :61-66)."""
    _need_cuda(score, label)
    score = score.detach().reshape(-1).float().contiguous()
    label = label.detach().reshape(-1).float().contiguous()
    n = score.numel()
    assert label.numel() == n, "auc: score / label size mismatch"
    out = torch.empty(3, dtype=torch.float64, device=score.device)
    nb = lib.twowl_auc_workspace_bytes(n)
    ws = _ws(nb, score.device)
    check(lib.twowl_auc(score.data_ptr(), label.data_ptr(), n, out.data_ptr(), ws.data_ptr(), nb, _stream()), "auc")
    _count(4 + 3 * 4)
    return out


RANK_MAX_K = 16   # TWOWL_RANK_MAX_K of include/twowl.h


def _rank_ks(ks):
    """The cut-off list as the host int64 array the ranking entry points take."""
    ks = [int(k) for k in ks]
    if not 1 <= len(ks) <= RANK_MAX_K or min(ks) < 1:
        raise ValueError(f"ks must hold 1..{RANK_MAX_K} cut-offs, each >= 1: {ks}")
    return (ctypes.c_int64 * len(ks))(*ks), len(ks)


def hits_at_k(score: torch.Tensor, label: torch.Tensor, ks) -> torch.Tensor:
    """Hits@K against a shared negative set on the device, OGB's _eval_hits (ogbl-collab, ogbl-ddi) -> float64[len(ks) + 2] =
    (hits@K for each K, n_pos, n_neg), no host sync. hits@K = fraction of the positives (label > 0.5) scored strictly above the
    K-th largest negative; 1.0 when there are fewer than K negatives; NaN when there is no positive or any score is NaN."""
    _need_cuda(score, label)
    score = score.detach().reshape(-1).float().contiguous()
    label = label.detach().reshape(-1).float().contiguous()
    n = score.numel()
    assert label.numel() == n, "hits_at_k: score / label size mismatch"
    h_ks, n_k = _rank_ks(ks)
    out = torch.empty(n_k + 2, dtype=torch.float64, device=score.device)
    nb = lib.twowl_hits_at_k_workspace_bytes(n)
    ws = _ws(nb, score.device)
    check(lib.twowl_hits_at_k(score.data_ptr(), label.data_ptr(), n, h_ks, n_k, out.data_ptr(), ws.data_ptr(), nb, _stream()),
          "hits_at_k")
    _count(5 + 3 * 4)
    return out


def rank_metrics(pos: torch.Tensor, neg: torch.Tensor, ks) -> torch.Tensor:
    """MRR and hits@k of each positive against its own negatives on the device, OGB's _eval_mrr (ogbl-citation2): pos [P],
    neg [P, k] -> float64[len(ks) + 2] = (MRR, hits@k for each k, P), no host sync. A positive's rank is 1 + the number of its
    negatives scored above it, ties counting half; NaN when P = 0 or any score is NaN. Two runs give the same bits."""
    _need_cuda(pos, neg)
    pos = pos.detach().reshape(-1).float().contiguous()
    P = pos.numel()
    assert neg.dim() == 2 and neg.shape[0] == P and neg.shape[1] >= 1, "rank_metrics: neg must be [P, k], k >= 1"
    k = neg.shape[1]
    neg = neg.detach().float().contiguous()
    h_ks, n_k = _rank_ks(ks)
    out = torch.empty(n_k + 2, dtype=torch.float64, device=pos.device)
    nb = lib.twowl_rank_metrics_workspace_bytes(P)
    ws = _ws(nb, pos.device)
    check(lib.twowl_rank_metrics(pos.data_ptr(), neg.data_ptr(), P, k, h_ks, n_k, out.data_ptr(), ws.data_ptr(), nb, _stream()),
          "rank_metrics")
    _count(3)
    return out


# ------------------------------------------------------------------------------ link-prediction heuristics

HEURISTICS = ("cn", "jaccard", "aa", "ra")   # the rows of link_heuristics


def simple_adjacency(row: torch.Tensor, col: torch.Tensor, num_nodes: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """The edges (row[e], col[e]) as an undirected simple graph -> (ptr int64 [N+1], adj int32 [nnz]): N(x) = adj[ptr[x]:ptr[x+1]]
    = every y != x joined to x by an edge in either direction, sorted ascending, each once. One host read (nnz and the bad-id
    count together); raises ValueError when an endpoint lies outside [0, num_nodes)."""
    _need_cuda(row, col)
    row, col = row.reshape(-1), col.reshape(-1)
    assert row.dtype == torch.int64 and col.dtype == torch.int64 and row.numel() == col.numel(), \
        "simple_adjacency: row / col must be int64 of one length"
    dev, E, n = row.device, row.numel(), int(num_nodes)
    ptr = torch.empty(n + 1, dtype=torch.int64, device=dev)
    adj = torch.empty(max(2 * E, 1), dtype=torch.int32, device=dev)
    bad = torch.empty(1, dtype=torch.int32, device=dev)
    nb = lib.twowl_simple_adjacency_workspace_bytes(E)
    ws = _ws(nb, dev)
    (pr, sr), (pc, sc) = (_row(row), _row(col)) if E else ((0, 1), (0, 1))
    check(lib.twowl_simple_adjacency(pr, sr, pc, sc, E, n, ptr.data_ptr(), adj.data_ptr(), bad.data_ptr(), ws.data_ptr(), nb,
                                     _stream()), "simple_adjacency")
    _count(6 + 2 * 3 * 3)
    nnz, nbad = torch.cat((ptr[n:], bad.to(torch.int64))).tolist()
    if nbad:
        raise ValueError(f"simple_adjacency: {nbad} edge endpoint(s) outside [0, {n})")
    return ptr, adj[:nnz].clone()


def link_heuristics(ptr: torch.Tensor, adj: torch.Tensor, u: torch.Tensor, v: torch.Tensor) -> torch.Tensor:
    """Neighbourhood scores of the query pairs (u[i], v[i]) over a simple adjacency (simple_adjacency) -> fp32 [4, P], rows in
    HEURISTICS order: common neighbours c = |N(u) ∩ N(v)|, Jaccard c / (d(u) + d(v) - c) (0 when that is 0), Adamic-Adar
    sum 1 / ln d(w) (terms with d(w) <= 1 count 0) and resource allocation sum 1 / d(w) over the common neighbours w. Bitwise
    repeatable and symmetric in (u, v). One host read; raises IndexError when a query id lies outside [0, N)."""
    _need_cuda(ptr, adj, u, v)
    assert ptr.dim() == 1 and ptr.dtype == torch.int64 and ptr.is_contiguous(), "link_heuristics: ptr must be contiguous int64 [N+1]"
    assert adj.dim() == 1 and adj.dtype == torch.int32 and adj.is_contiguous(), "link_heuristics: adj must be contiguous int32"
    u, v = u.reshape(-1).to(torch.int64), v.reshape(-1).to(torch.int64)
    assert u.numel() == v.numel(), "link_heuristics: u / v size mismatch"
    dev, n, P = ptr.device, ptr.numel() - 1, u.numel()
    (pu, su), (pv, sv) = (_row(u), _row(v)) if P else ((0, 1), (0, 1))
    chunk_off = torch.empty(P + 1, dtype=torch.int64, device=dev)
    info = torch.empty(3, dtype=torch.int64, device=dev)
    nb = lib.twowl_link_plan_workspace_bytes(P)
    ws = _ws(nb, dev)
    check(lib.twowl_link_plan(ptr.data_ptr(), n, pu, su, pv, sv, P, chunk_off.data_ptr(), info.data_ptr(), ws.data_ptr(), nb,
                              _stream()), "link_plan")
    nbad, n_chunks, _ = info.tolist()
    if nbad:
        raise IndexError(f"link_heuristics: {nbad} query id(s) outside [0, {n})")
    out = torch.empty((4, P), dtype=torch.float32, device=dev)
    nb = lib.twowl_link_heuristics_workspace_bytes(n_chunks)
    ws = _ws(nb, dev)
    check(lib.twowl_link_heuristics(ptr.data_ptr(), adj.data_ptr(), n, pu, su, pv, sv, P, chunk_off.data_ptr(), n_chunks,
                                    out.data_ptr(), ws.data_ptr(), nb, _stream()), "link_heuristics")
    _count(5 + 2)
    return out


def _scan_launches(n: int) -> int:
    """Launches of one scan_exclusive_i64 over n values: three kernels, or one memset when n is 0."""
    return 3 if n > 0 else 1


class CommonNeighbors:
    """The common neighbours of a batch of query pairs (common_neighbors), as a CSR by pair: ptr int64 [P+1], ids int32 [nnz] (row p =
    CN(p) in ascending id order) and pair int32 [nnz] (each entry's pair, nondecreasing: what a backward by node needs)."""
    __slots__ = ("ptr", "ids", "pair")

    def __init__(self, ptr, ids, pair):
        self.ptr, self.ids, self.pair = ptr, ids, pair

    @property
    def num_pairs(self) -> int:
        return self.ptr.numel() - 1


def _check_adjacency(fn: str, ptr, adj):
    assert ptr.dim() == 1 and ptr.dtype == torch.int64 and ptr.is_contiguous(), f"{fn}: ptr must be contiguous int64 [N+1]"
    assert adj.dim() == 1 and adj.dtype == torch.int32 and adj.is_contiguous(), f"{fn}: adj must be contiguous int32"


def adjacency_pair_mask(ptr: torch.Tensor, adj: torch.Tensor, u: torch.Tensor, v: torch.Tensor) -> torch.Tensor:
    """uint8 [nnz] over a simple adjacency (simple_adjacency): 1 at the entries of v in N(u) and of u in N(v) for every pair (u[i],
    v[i]) that is an edge - the mask that deletes those edges for common_neighbors. Non-edges and u == v set nothing. One host
    read; raises IndexError when an id lies outside [0, N)."""
    _need_cuda(ptr, adj, u, v)
    _check_adjacency("adjacency_pair_mask", ptr, adj)
    u, v = u.reshape(-1).to(torch.int64), v.reshape(-1).to(torch.int64)
    assert u.numel() == v.numel(), "adjacency_pair_mask: u / v size mismatch"
    dev, n, P = ptr.device, ptr.numel() - 1, u.numel()
    (pu, su), (pv, sv) = (_row(u), _row(v)) if P else ((0, 1), (0, 1))
    mask = torch.empty(adj.numel(), dtype=torch.uint8, device=dev)
    info = torch.empty(1, dtype=torch.int64, device=dev)
    check(lib.twowl_adjacency_pair_mask(ptr.data_ptr(), adj.data_ptr(), n, adj.numel(), pu, su, pv, sv, P, mask.data_ptr(),
                                        info.data_ptr(), _stream()), "adjacency_pair_mask")
    _count(1 + int(adj.numel() > 0) + int(P > 0))
    nbad = int(info.item())
    if nbad:
        raise IndexError(f"adjacency_pair_mask: {nbad} id(s) outside [0, {n})")
    return mask


def common_neighbors(ptr: torch.Tensor, adj: torch.Tensor, u: torch.Tensor, v: torch.Tensor,
                     entry_mask: Optional[torch.Tensor] = None) -> CommonNeighbors:
    """The common neighbours CN(i) = N(u[i]) ∩ N(v[i]) of each query pair over a simple adjacency (simple_adjacency) ->
    CommonNeighbors. entry_mask (uint8 [nnz], e.g. adjacency_pair_mask) deletes the adjacency entries it marks. u == v gives N(u).
    The pairs are cut as link_heuristics cuts them, |CN(i)| equals its cn row, and the lists are bitwise repeatable. Two host
    reads (the plan, the total); raises IndexError when an id lies outside [0, N) and ValueError when the lists would hold
    2^31 or more entries (split the query list)."""
    fn = "common_neighbors"
    _need_cuda(ptr, adj, u, v, entry_mask)
    _check_adjacency(fn, ptr, adj)
    if entry_mask is not None:
        assert entry_mask.dtype == torch.uint8 and entry_mask.is_contiguous() and entry_mask.numel() == adj.numel(), \
            f"{fn}: entry_mask must be contiguous uint8 [nnz]"
    u, v = u.reshape(-1).to(torch.int64), v.reshape(-1).to(torch.int64)
    assert u.numel() == v.numel(), f"{fn}: u / v size mismatch"
    dev, n, P = ptr.device, ptr.numel() - 1, u.numel()
    (pu, su), (pv, sv) = (_row(u), _row(v)) if P else ((0, 1), (0, 1))
    chunk_off = torch.empty(P + 1, dtype=torch.int64, device=dev)
    info = torch.empty(3, dtype=torch.int64, device=dev)
    nb = lib.twowl_link_plan_workspace_bytes(P)
    ws = _ws(nb, dev)
    check(lib.twowl_link_plan(ptr.data_ptr(), n, pu, su, pv, sv, P, chunk_off.data_ptr(), info.data_ptr(), ws.data_ptr(), nb,
                              _stream()), "link_plan")
    _count(1 + int(P > 0) + _scan_launches(P))
    nbad, n_chunks, _ = info.tolist()
    if nbad:
        raise IndexError(f"{fn}: {nbad} query id(s) outside [0, {n})")
    cn_ptr = torch.empty(P + 1, dtype=torch.int64, device=dev)
    chunk_base = torch.empty(n_chunks + 1, dtype=torch.int64, device=dev)
    nb = lib.twowl_common_neighbors_count_workspace_bytes(P, n_chunks)
    ws = _ws(nb, dev)
    mp = _p(entry_mask)
    check(lib.twowl_common_neighbors_count(ptr.data_ptr(), adj.data_ptr(), n, mp, pu, su, pv, sv, P, chunk_off.data_ptr(), n_chunks,
                                           cn_ptr.data_ptr(), chunk_base.data_ptr(), ws.data_ptr(), nb, _stream()),
          "common_neighbors_count")
    _count(int(n_chunks > 0) + int(P > 0) + _scan_launches(P) + _scan_launches(n_chunks))
    total = int(cn_ptr[P].item())
    if total >= 2 ** 31:
        raise ValueError(f"{fn}: the lists would hold {total} >= 2^31 entries; pass fewer pairs per call")
    ids = torch.empty(total, dtype=torch.int32, device=dev)
    pair = torch.empty(total, dtype=torch.int32, device=dev)
    check(lib.twowl_common_neighbors_fill(ptr.data_ptr(), adj.data_ptr(), n, mp, pu, su, pv, sv, P, chunk_off.data_ptr(), n_chunks,
                                          cn_ptr.data_ptr(), chunk_base.data_ptr(), total, _p(ids) if total else None,
                                          _p(pair) if total else None, _stream()), "common_neighbors_fill")
    _count((int(n_chunks > 0) + 1) if total else 0)
    return CommonNeighbors(cn_ptr, ids, pair)


SKETCH_MAX_HOPS = 3      # TWOWL_SKETCH_MAX_HOPS of include/twowl.h
SKETCH_CHUNK = 64        # rows of the adjacency longer than this are cut into chunks of this many entries (any value gives the same bits)


class LinkSketches:
    """BUDDY's per-node sketches of the d-hop neighbourhoods N_{<=d}(x), d = 0 .. hops (link_sketches): minhash int32 [hops+1, N,
    num_perm] (uint32 bits) and hll uint8 [hops+1, N, 2^hll_p], with the parameters they were built with."""
    __slots__ = ("minhash", "hll", "hops", "num_perm", "hll_p", "seed")

    def __init__(self, minhash, hll, hops, num_perm, hll_p, seed):
        self.minhash, self.hll, self.hops, self.num_perm, self.hll_p, self.seed = minhash, hll, hops, num_perm, hll_p, seed

    @property
    def num_nodes(self) -> int:
        return self.minhash.shape[1]

    @property
    def num_features(self) -> int:
        return self.hops * self.hops + 2 * self.hops


def _sketch_params(fn: str, hops: int, num_perm: int, hll_p: int):
    if not 1 <= int(hops) <= SKETCH_MAX_HOPS:
        raise ValueError(f"{fn}: hops = {hops} outside [1, {SKETCH_MAX_HOPS}]")
    if not (32 <= int(num_perm) <= 1024 and int(num_perm) % 32 == 0):
        raise ValueError(f"{fn}: num_perm = {num_perm} must be a multiple of 32 in [32, 1024]")
    if not 4 <= int(hll_p) <= 10:
        raise ValueError(f"{fn}: hll_p = {hll_p} outside [4, 10]")


def link_sketches(ptr: torch.Tensor, adj: torch.Tensor, hops: int = 2, num_perm: int = 128, hll_p: int = 8, seed: int = 0,
                  entry_mask: Optional[torch.Tensor] = None, chunk: int = SKETCH_CHUNK) -> LinkSketches:
    """BUDDY's MinHash and HyperLogLog sketches of every node's d-hop neighbourhood, d = 0 .. hops, over a simple adjacency
    (simple_adjacency) -> LinkSketches. Hop 0 sketches {x} (twowl_sketch_init defines the hashes from seed); hop d is the elementwise
    min (MinHash) and bytewise max (HyperLogLog) of x's hop d-1 row and those of its neighbours. entry_mask (uint8 [nnz], e.g.
    adjacency_pair_mask) deletes the adjacency entries it marks. chunk only sets how a long row is cut: the bits never depend on it.
    No host read."""
    fn = "link_sketches"
    _need_cuda(ptr, adj, entry_mask)
    _check_adjacency(fn, ptr, adj)
    _sketch_params(fn, hops, num_perm, hll_p)
    if not 1 <= int(chunk) <= 1 << 30:
        raise ValueError(f"{fn}: chunk = {chunk} outside [1, 2^30]")
    if entry_mask is not None:
        assert entry_mask.dtype == torch.uint8 and entry_mask.is_contiguous() and entry_mask.numel() == adj.numel(), \
            f"{fn}: entry_mask must be contiguous uint8 [nnz]"
    hops, num_perm, hll_p, seed = int(hops), int(num_perm), int(hll_p), int(seed) % (2 ** 64)
    dev, n, nnz, m = ptr.device, ptr.numel() - 1, adj.numel(), 1 << int(hll_p)
    mh = torch.empty((hops + 1, n, num_perm), dtype=torch.int32, device=dev)
    hll = torch.empty((hops + 1, n, m), dtype=torch.uint8, device=dev)
    check(lib.twowl_sketch_init(n, num_perm, hll_p, seed, mh.data_ptr(), hll.data_ptr(), _stream()), "sketch_init")
    _count(int(n > 0))
    nb = lib.twowl_sketch_hop_workspace_bytes(nnz, num_perm, hll_p, int(chunk))
    ws = _ws(nb, dev)
    for d in range(1, hops + 1):
        with _P("sketch_hop", (nnz + n) * (4 * num_perm + m) + n * (4 * num_perm + m)):
            check(lib.twowl_sketch_hop(ptr.data_ptr(), _p(adj) if nnz else None, n, nnz, _p(entry_mask), num_perm, hll_p, int(chunk),
                                       mh[d - 1].data_ptr(), hll[d - 1].data_ptr(), mh[d].data_ptr(), hll[d].data_ptr(),
                                       ws.data_ptr(), nb, _stream()), "sketch_hop")
        _count(5 if n else 0)
    return LinkSketches(mh, hll, hops, num_perm, hll_p, seed)


def sketch_features(sk: LinkSketches, u: torch.Tensor, v: torch.Tensor) -> torch.Tensor:
    """BUDDY's structure features of the pairs (u[i], v[i]) from their sketches (link_sketches) -> fp32 [P, hops^2 + 2 hops]:
    the estimated counts A(d1, d2) of nodes at distance exactly d1 from u and d2 from v (row-major over d1, d2 = 1 .. hops), then
    B_u(d) and B_v(d), the nodes at distance d from one endpoint and more than hops from the other (include/twowl.h restates the
    estimators). One host read; raises IndexError when an id lies outside [0, N)."""
    fn = "sketch_features"
    _need_cuda(sk.minhash, sk.hll, u, v)
    _sketch_params(fn, sk.hops, sk.num_perm, sk.hll_p)
    u, v = u.reshape(-1).to(torch.int64), v.reshape(-1).to(torch.int64)
    assert u.numel() == v.numel(), f"{fn}: u / v size mismatch"
    dev, n, P = sk.minhash.device, sk.num_nodes, u.numel()
    (pu, su), (pv, sv) = (_row(u), _row(v)) if P else ((0, 1), (0, 1))
    out = torch.empty((P, sk.num_features), dtype=torch.float32, device=dev)
    info = torch.empty(1, dtype=torch.int64, device=dev)
    check(lib.twowl_sketch_pair_features(sk.hops, n, sk.num_perm, sk.hll_p, sk.minhash.data_ptr(), sk.hll.data_ptr(), pu, su, pv, sv, P,
                                         out.data_ptr(), info.data_ptr(), _stream()), "sketch_pair_features")
    _count(1 + int(P > 0))
    nbad = int(info.item())
    if nbad:
        raise IndexError(f"{fn}: {nbad} pair(s) with an id outside [0, {n})")
    return out


RECOMMEND_MAX_ENTRIES = 1 << 26   # default expansion budget of one batch: 44 B of workspace per entry, about 3 GB


def _sort_launches(bits: int) -> int:
    """Launches of one radix_sort_pairs: histogram, 3-kernel scan and scatter per 8-bit pass, two copies after an even count."""
    p = max(1, (max(1, bits) + 7) // 8)
    return 5 * p + 2 * (1 - p % 2)


def recommend_links(ptr: torch.Tensor, adj: torch.Tensor, src: torch.Tensor, k: int, by: str = "aa",
                    max_entries: Optional[int] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Each source's top-k link candidates over a simple adjacency (simple_adjacency) -> (ids int64 [Q, k], scores fp32 [4, Q, k]).

    The candidates of s are its two-hop non-neighbours {v != s : v not in N(s), N(s) ∩ N(v) non-empty}; any other node scores 0
    under every heuristic. Row q holds the top min(k, #candidates) of src[q] ordered by the heuristic `by` (one of HEURISTICS)
    descending, ties by id ascending, then -1 ids and NaN scores. scores[j] is heuristic HEURISTICS[j] of each returned pair, as
    link_heuristics defines it, except that aa and ra are summed in double over the common neighbours in ascending id order, one
    at a time: a sequential numpy sum reproduces cn, jaccard and ra bit for bit.

    The work of a source is its expansion X(s) = sum of d(w) over w in N(s). The queries run in consecutive batches of at most
    max_entries expansion entries (default RECOMMEND_MAX_ENTRIES); a source that expands to more runs alone. The result is
    bitwise repeatable and does not depend on max_entries. One host read (the plan); raises IndexError when a source id lies
    outside [0, N) and ValueError for an unknown `by` or k < 1."""
    if by not in HEURISTICS:
        raise ValueError(f"recommend_links: by must be one of {HEURISTICS}, got {by!r}")
    k = int(k)
    if k < 1:
        raise ValueError(f"recommend_links: k must be >= 1, got {k}")
    budget = RECOMMEND_MAX_ENTRIES if max_entries is None else max(1, int(max_entries))
    _need_cuda(ptr, adj, src)
    assert ptr.dim() == 1 and ptr.dtype == torch.int64 and ptr.is_contiguous(), "recommend_links: ptr must be contiguous int64 [N+1]"
    assert adj.dim() == 1 and adj.dtype == torch.int32 and adj.is_contiguous(), "recommend_links: adj must be contiguous int32"
    src = src.reshape(-1).to(torch.int64)
    dev, n, Q = ptr.device, ptr.numel() - 1, src.numel()
    ps, ss = _row(src) if Q else (0, 1)
    exp_off = torch.empty(Q + 1, dtype=torch.int64, device=dev)
    info = torch.empty(2, dtype=torch.int64, device=dev)
    nb = lib.twowl_recommend_plan_workspace_bytes(Q)
    ws = _ws(nb, dev)
    check(lib.twowl_recommend_plan(ptr.data_ptr(), adj.data_ptr(), n, ps, ss, Q, exp_off.data_ptr(), info.data_ptr(), ws.data_ptr(),
                                   nb, _stream()), "recommend_plan")
    _count(6)
    host = torch.cat((info, exp_off)).cpu().numpy()
    if host[0]:
        raise IndexError(f"recommend_links: {int(host[0])} source id(s) outside [0, {n})")
    off = host[2:]
    batches, q = [], 0
    while q < Q:   # consecutive queries while the expansion stays within the budget; at least one query per batch
        e = min(Q, max(q + 1, int(np.searchsorted(off, off[q] + budget, side="right")) - 1))
        batches.append((q, e, int(off[e] - off[q])))
        q = e
    ids = torch.empty((Q, k), dtype=torch.int64, device=dev)
    scores = torch.empty((4, Q, k), dtype=torch.float32, device=dev)
    if not batches:
        return ids, scores
    nb = lib.twowl_recommend_workspace_bytes(max(b[2] for b in batches), max(b[1] - b[0] for b in batches))
    ws = _ws(nb, dev)
    j_by = HEURISTICS.index(by)
    for q0, q1, m in batches:
        check(lib.twowl_recommend(ptr.data_ptr(), adj.data_ptr(), n, ps, ss, Q, q0, q1, exp_off.data_ptr(), m, j_by, k, ids.data_ptr(),
                                  scores.data_ptr(), ws.data_ptr(), nb, _stream()), "recommend")
        if m:   # expansion (9 launches), three small kernels between and after the four sorts
            qb = q1 - q0
            _count(12 + _sort_launches((n - 1).bit_length()) + _sort_launches((qb - 1).bit_length()) + _sort_launches(32)
                   + _sort_launches(qb.bit_length()))
        _count(1)
    return ids, scores


# ------------------------------------------------------------------------------ global link-prediction heuristics

GLOBAL_HEURISTICS = ("katz", "ppr")
GLOBAL_DEFAULTS = {"katz": (3, 0.001), "ppr": (20, 0.85)}   # (steps, damping): SEAL's beta and alpha
WALK_MAX_COLS = 256      # default sources per batch: the operand pair is 2 x N x 256 x 4 bytes, 2 GB at N = 1 M (DESIGN.md §0)
# seg_reduce hands a row of more than 32 chunks to a whole CTA whose lane-group count depends on the operand width up to 68
# columns and is fixed from there on: an operand of at least 68 columns gives every column the same bits at every batch width
_WALK_MIN_WIDTH = 68
_WALK_MAX_WIDTH = 1024   # seg_reduce's widest operand


def _walk_params(fn: str, by: str, steps, damping) -> Tuple[int, float]:
    if by not in GLOBAL_HEURISTICS:
        raise ValueError(f"{fn}: by must be one of {GLOBAL_HEURISTICS}, got {by!r}")
    d_steps, d_damp = GLOBAL_DEFAULTS[by]
    steps = d_steps if steps is None else int(steps)
    if steps < 1:
        raise ValueError(f"{fn}: steps must be >= 1, got {steps}")
    with np.errstate(over="ignore"):     # the recursion runs on the fp32-rounded parameter; one that overflows fp32 is refused
        damp = float(np.float32(d_damp if damping is None else damping))
    if by == "katz" and not (np.isfinite(damp) and damp > 0):
        raise ValueError(f"{fn}: the Katz damping beta must be finite and > 0, got {damping}")
    if by == "ppr" and not 0 < damp < 1:
        raise ValueError(f"{fn}: the PageRank damping alpha must lie in (0, 1), got {damping}")
    return steps, damp


def _walk_cols(fn: str, max_cols) -> int:
    b = WALK_MAX_COLS if max_cols is None else int(max_cols)
    if not 1 <= b <= _WALK_MAX_WIDTH:
        raise ValueError(f"{fn}: max_cols must lie in [1, {_WALK_MAX_WIDTH}], got {b}")
    return b


class _Walk:
    """The operands of batched walks from up to `cols` sources over a simple adjacency: two fp32 [N, ld] buffers, ld the batch
    width rounded up to a multiple of 4 and at least _WALK_MIN_WIDTH (columns past a batch's sources stay 0), the long-row plan
    and the per-node scale."""

    def __init__(self, ptr, adj, by: str, steps: int, damping: float, cols: int):
        n, dev = ptr.numel() - 1, ptr.device
        self.ptr, self.adj, self.n, self.by, self.steps, self.damping = ptr, adj, n, by, steps, damping
        self.ld = min(_WALK_MAX_WIDTH, max(_WALK_MIN_WIDTH, -(-cols // 4) * 4))
        self.Y = [torch.empty((n, self.ld), dtype=torch.float32, device=dev) for _ in range(2)]
        self.plan = seg_plan(ptr, n, adj.numel())
        self.scale = torch.empty(n, dtype=torch.float32, device=dev)
        check(lib.twowl_walk_scale(ptr.data_ptr(), n, int(by == "ppr"), damping, self.scale.data_ptr(), _stream()), "walk_scale")
        _count()

    def _restart(self, Y, src, n_cols: int, value: float):
        ps, ss = _row(src)
        check(lib.twowl_walk_restart(Y.data_ptr(), self.ld, self.n, ps, ss, n_cols, value, _stream()), "walk_restart")
        _count()

    def run(self, src: torch.Tensor) -> torch.Tensor:
        """Scores of every node from each source of src (int64, at most ld ids, all valid) -> Y: column j for src[j]."""
        Y, Z = self.Y
        Y.zero_()
        n_cols = src.numel()
        ppr = self.by == "ppr"
        if ppr:
            self._restart(Y, src, n_cols, 1.0)
        for _ in range(self.steps):
            if not ppr:
                self._restart(Y, src, n_cols, 1.0)
            seg_reduce(self.ptr, self.adj, self.n, Y, plan=self.plan, src_scale=self.scale, out=Z)
            if ppr:
                self._restart(Z, src, n_cols, float(np.float32(1) - np.float32(self.damping)))
            Y, Z = Z, Y
        self.Y = [Y, Z]
        return Y


def _check_graph(fn: str, ptr, adj):
    assert ptr.dim() == 1 and ptr.dtype == torch.int64 and ptr.is_contiguous(), f"{fn}: ptr must be contiguous int64 [N+1]"
    assert adj.dim() == 1 and adj.dtype == torch.int32 and adj.is_contiguous(), f"{fn}: adj must be contiguous int32"


def global_heuristics(ptr: torch.Tensor, adj: torch.Tensor, u: torch.Tensor, v: torch.Tensor, by: str = "katz", steps: Optional[int] = None,
                      damping: Optional[float] = None, max_cols: Optional[int] = None) -> torch.Tensor:
    """Global (path-based) scores of the query pairs (u[i], v[i]) over a simple adjacency (simple_adjacency) -> fp32 [P], each
    rooted at its first endpoint u[i]:
      by="katz": sum_{l=1..steps} beta^l (A^l)[u, v], truncated Katz (default steps 3, beta = damping = 0.001);
      by="ppr":  pi_steps[v] of personalized PageRank from u: pi_0 = e_u, pi_{t+1} = alpha A D^-1 pi_t + (1 - alpha) e_u (default
                 steps 20, alpha = damping = 0.85); mass at an isolated node is dropped.
    Everything runs in fp32 with the fp32-rounded damping. Katz is symmetric in exact arithmetic, but the fp32 scores of (u, v) and
    (v, u) come from different walks and may differ in the last bits; PPR is not symmetric. A score whose paths all underflow
    fp32 (PPR through hubs: (1 / d)^steps) is 0.

    The distinct u are the walks' sources, up to max_cols (default WALK_MAX_COLS, at most 1024) per batch; each batch is `steps`
    seg_reduce passes over the adjacency on an [N, max(68, max_cols)] operand. The result is bitwise repeatable and does not depend
    on max_cols. One host read (the bad-id count and the number of distinct u); raises IndexError for an id outside [0, N) and
    ValueError for an unknown `by`, steps < 1, a Katz damping that is not finite and > 0 or a PageRank damping outside (0, 1)."""
    steps, damp = _walk_params("global_heuristics", by, steps, damping)
    cols = _walk_cols("global_heuristics", max_cols)
    _need_cuda(ptr, adj, u, v)
    _check_graph("global_heuristics", ptr, adj)
    u, v = u.reshape(-1).to(torch.int64), v.reshape(-1).to(torch.int64)
    assert u.numel() == v.numel(), "global_heuristics: u / v size mismatch"
    dev, n, P = ptr.device, ptr.numel() - 1, u.numel()
    out = torch.empty(P, dtype=torch.float32, device=dev)
    if P == 0:
        return out
    # the pairs ordered by source once; column c = rank of the source among the distinct u
    us, order = torch.sort(u, stable=True)
    new = torch.ones(P, dtype=torch.bool, device=dev)
    new[1:] = us[1:] != us[:-1]
    col = torch.cumsum(new, 0) - 1
    bad = ((u < 0) | (u >= n) | (v < 0) | (v >= n)).sum()
    nbad, U = torch.stack((bad, col[-1] + 1)).tolist()
    if nbad:
        raise IndexError(f"global_heuristics: {nbad} query id(s) outside [0, {n})")
    sources = torch.zeros(P, dtype=torch.int64, device=dev).scatter_(0, col, us)[:U]
    vs = v[order].contiguous()
    walk = _Walk(ptr, adj, by, steps, damp, min(cols, U))
    for c0 in range(0, U, cols):
        c1 = min(U, c0 + cols)
        Y = walk.run(sources[c0:c1])
        check(lib.twowl_walk_gather(Y.data_ptr(), walk.ld, n, col.data_ptr(), vs.data_ptr(), order.data_ptr(), P, c0, c1, out.data_ptr(),
                                    _stream()), "walk_gather")
        _count()
    return out


def recommend_global(ptr: torch.Tensor, adj: torch.Tensor, src: torch.Tensor, k: int, by: str = "ppr", steps: Optional[int] = None,
                     damping: Optional[float] = None, max_cols: Optional[int] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Each source's top-k link candidates by a global heuristic (see global_heuristics) -> (ids int64 [Q, k], scores fp32 [Q, k]).

    The candidates of s are {v != s : v not in N(s), score(s, v) > 0}, at any distance: every node a walk of at most `steps` edges
    reaches (Katz), or that keeps an fp32 share of the walk's mass (PPR). Row q holds the top min(k, #candidates) of src[q] by score
    descending, ties by id ascending, then -1 ids and NaN scores. scores[q, j] is bit-identical to
    global_heuristics(src[q], ids[q, j]) with the same parameters. One walk per query, in src order, max_cols per batch (duplicates
    are walked again); the result is bitwise repeatable and independent of max_cols. One host read (the bad-id count); raises
    IndexError for a source outside [0, N) and ValueError as global_heuristics does or for k < 1."""
    steps, damp = _walk_params("recommend_global", by, steps, damping)
    cols = _walk_cols("recommend_global", max_cols)
    k = int(k)
    if k < 1:
        raise ValueError(f"recommend_global: k must be >= 1, got {k}")
    _need_cuda(ptr, adj, src)
    _check_graph("recommend_global", ptr, adj)
    src = src.reshape(-1).to(torch.int64)
    dev, n, Q = ptr.device, ptr.numel() - 1, src.numel()
    ids = torch.empty((Q, k), dtype=torch.int64, device=dev)
    scores = torch.empty((Q, k), dtype=torch.float32, device=dev)
    if Q == 0:
        return ids, scores
    nbad = int(((src < 0) | (src >= n)).sum())
    if nbad:
        raise IndexError(f"recommend_global: {nbad} source id(s) outside [0, {n})")
    walk = _Walk(ptr, adj, by, steps, damp, min(cols, Q))
    nb = lib.twowl_walk_topk_workspace_bytes(n, min(cols, Q), k)
    ws = _ws(nb, dev)
    kk = min(k, n)
    for q0 in range(0, Q, cols):
        q1 = min(Q, q0 + cols)
        Y = walk.run(src[q0:q1])
        ps, ss = _row(src[q0:q1])
        check(lib.twowl_walk_topk(ptr.data_ptr(), adj.data_ptr(), n, Y.data_ptr(), walk.ld, ps, ss, q1 - q0, k, Q, q0, ids.data_ptr(),
                                  scores.data_ptr(), ws.data_ptr(), nb, _stream()), "walk_topk")
        if kk:   # exclusion, memset, 4 x (histogram, select), count, scan, take, scan, write, two sorts with a key kernel between
            _count(1 + 1 + 8 + 1 + 3 + 1 + 3 + 1 + _sort_launches(32) + 1 + _sort_launches((q1 - q0 - 1).bit_length()))
        _count(1)
    return ids, scores


# ------------------------------------------------------------------------------ node2vec

N2V_MAX_RATIO = 1024.0   # max(1/p, 1, 1/q) / min(1/p, 1, 1/q): the expected number of rejection trials per walk step
N2V_MAX_DIM = 512


def _n2v_pq(fn: str, p, q) -> Tuple[float, float]:
    p, q = float(p), float(q)
    if not (np.isfinite(p) and np.isfinite(q) and p > 0 and q > 0):
        raise ValueError(f"{fn}: p and q must be finite and > 0, got p={p}, q={q}")
    w = (1.0 / p, 1.0, 1.0 / q)
    if max(w) / min(w) > N2V_MAX_RATIO:
        raise ValueError(f"{fn}: max(1/p, 1, 1/q) / min(1/p, 1, 1/q) must be <= {N2V_MAX_RATIO:g} (the expected rejection trials "
                         f"per step), got p={p}, q={q}")
    return p, q


def _n2v_dim(fn: str, d: int) -> int:
    d = int(d)
    if d < 32 or d > N2V_MAX_DIM or d % 32:
        raise ValueError(f"{fn}: the embedding width must be a multiple of 32 in [32, {N2V_MAX_DIM}], got {d}")
    return d


def _n2v_walks(ptr, adj, start, length: int, p: float, q: float, seed: int, index_base: int) -> torch.Tensor:
    """The launch of node2vec_walks without its checks (start int64 1-D, every id valid)."""
    W, n = start.numel(), ptr.numel() - 1
    walks = torch.empty((W, length), dtype=torch.int32, device=ptr.device)
    if W == 0:
        return walks
    ps, ss = _row(start)
    check(lib.twowl_n2v_walks(ptr.data_ptr(), adj.data_ptr(), n, ps, ss, W, length, p, q, seed & (2 ** 64 - 1), index_base,
                              walks.data_ptr(), _stream()), "n2v_walks")
    _count()
    return walks


def node2vec_walks(ptr: torch.Tensor, adj: torch.Tensor, start: torch.Tensor, length: int, p: float = 1.0, q: float = 1.0,
                   seed: Optional[int] = None, index_base: int = 0) -> torch.Tensor:
    """node2vec's second-order biased random walks over a simple adjacency (simple_adjacency) -> int32 [W, length], row i the walk
    from start[i]. The first step is uniform over N(start); after it, from cur with predecessor prev, the next node x in N(cur) is
    drawn with probability proportional to 1/p if x == prev, 1 if x is a neighbour of prev and 1/q otherwise (node2vec's transition
    rule for an unweighted graph). A walk from an isolated start is [s, -1, -1, ...].

    Sampling is by rejection (KnightKing): x is proposed uniformly from N(cur), a 32-bit multiply-high whose bias is at most
    d(cur) / 2^32, and accepted with probability w(x) / max(w); p = q = 1 accepts every proposal (DeepWalk). The draws are
    counter-based, keyed by (seed, index_base + i, step, trial), so a walk depends on (seed, index_base + i, start[i]) alone:
    node2vec_walks(.., start, base=0)[a:b] equals node2vec_walks(.., start[a:b], base=a) bit for bit. seed=None takes next_seed().
    One host read (the bad-id count); raises IndexError for a start outside [0, N) and ValueError for length < 1 or p, q that are
    not finite and > 0 or whose weight ratio max(w) / min(w) exceeds N2V_MAX_RATIO (the expected trials per step)."""
    p, q = _n2v_pq("node2vec_walks", p, q)
    length = int(length)
    if length < 1:
        raise ValueError(f"node2vec_walks: length must be >= 1, got {length}")
    index_base = int(index_base)
    if index_base < 0:
        raise ValueError(f"node2vec_walks: index_base must be >= 0, got {index_base}")
    _need_cuda(ptr, adj, start)
    _check_graph("node2vec_walks", ptr, adj)
    start = start.reshape(-1).to(torch.int64)
    n = ptr.numel() - 1
    if start.numel():
        nbad = int(((start < 0) | (start >= n)).sum())
        if nbad:
            raise IndexError(f"node2vec_walks: {nbad} start id(s) outside [0, {n})")
    return _n2v_walks(ptr, adj, start, length, p, q, next_seed() if seed is None else int(seed), index_base)


def _n2v_step(emb, exp_avg, exp_avg_sq, step, walks, negs, window: int, lr: float, betas, eps: float) -> torch.Tensor:
    """The launch of node2vec_step without its id check."""
    n, d = emb.shape
    B, L = walks.shape
    K = negs.shape[2]
    loss = torch.empty((), dtype=torch.float64, device=emb.device)
    nb = lib.twowl_n2v_step_workspace_bytes(B, L, window, K, d)
    ws = _ws(nb, emb.device)
    check(lib.twowl_n2v_step(emb.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(), step.data_ptr(), n, d, walks.data_ptr(),
                             negs.data_ptr(), B, L, window, K, float(lr), float(betas[0]), float(betas[1]), float(eps), loss.data_ptr(),
                             ws.data_ptr(), nb, _stream()), "n2v_step")
    _count(1 + (9 + _sort_launches(max(1, n).bit_length()) + 3 if B * L else 0) + 1)
    return loss


def _n2v_step_args(emb, exp_avg, exp_avg_sq, step, walks, negs, window):
    _need_cuda(emb, exp_avg, exp_avg_sq, step, walks, negs)
    assert emb.dim() == 2 and all(t.dtype == torch.float32 and t.is_contiguous() and t.shape == emb.shape for t in (emb, exp_avg, exp_avg_sq)), \
        "node2vec_step: emb / exp_avg / exp_avg_sq must be contiguous fp32 [N, d] of one shape"
    assert step.dtype == torch.int64 and step.numel() == 1, "node2vec_step: step must be an int64 device scalar"
    assert walks.dim() == 2 and walks.dtype == torch.int32 and walks.is_contiguous(), "node2vec_step: walks must be contiguous int32 [B, L]"
    assert negs.dim() == 3 and negs.dtype == torch.int32 and negs.is_contiguous() and negs.shape[:2] == walks.shape, \
        "node2vec_step: negs must be contiguous int32 [B, L, K]"
    _n2v_dim("node2vec_step", emb.shape[1])
    window = int(window)
    if window < 1:
        raise ValueError(f"node2vec_step: window must be >= 1, got {window}")
    if negs.shape[2] < 1:
        raise ValueError("node2vec_step: negs must hold K >= 1 negatives per token")
    return window


def node2vec_step(emb: torch.Tensor, exp_avg: torch.Tensor, exp_avg_sq: torch.Tensor, step: torch.Tensor, walks: torch.Tensor,
                  negs: torch.Tensor, window: int, lr: float = 0.01, betas=(0.9, 0.999), eps: float = 1e-8) -> torch.Tensor:
    """One skip-gram step with negative sampling on the embedding table emb (fp32 [N, d], d a multiple of 32 up to 512), in place,
    with lazy Adam -> the loss, a 0-dim float64 device tensor (no host read).

    Positive pairs are (walks[b, i], walks[b, i + o]) for 1 <= o <= window, i + o < L, both entries >= 0 (walks int32 [B, L], -1
    padding); negative pairs are (walks[b, i], negs[b, i, j]) for every j < K (negs int32 [B, L, K]) of each token i with at least
    one positive pair; self pairs are kept. Loss = mean_pos softplus(-e_a . e_b) + mean_neg softplus(e_a . e_b) (PyG Node2Vec's
    objective). The rows in any pair are updated exactly as torch.optim.SparseAdam updates the coalesced gradient of an
    nn.Embedding(sparse=True), the gradient taken from the table before the step: exp_avg, exp_avg_sq and the int64 device scalar
    `step` (the step count, advanced only when the batch has a positive pair) are the optimiser state. No other row changes; a
    batch without a positive pair changes nothing and its loss is 0. Bitwise repeatable. One host read (the id check); raises
    IndexError for an id outside [-1, N) in walks or [0, N) in negs and ValueError for d, window < 1 or K < 1."""
    window = _n2v_step_args(emb, exp_avg, exp_avg_sq, step, walks, negs, window)
    n = emb.shape[0]
    if walks.numel():
        bad = ((walks < -1) | (walks >= n)).sum()
        if negs.numel():
            bad = bad + ((negs < 0) | (negs >= n)).sum()
        nbad = int(bad)
        if nbad:
            raise IndexError(f"node2vec_step: {nbad} id(s) outside [-1, {n}) in walks or [0, {n}) in negs")
    return _n2v_step(emb, exp_avg, exp_avg_sq, step, walks, negs, window, lr, betas, eps)


def embedding_dot(emb: torch.Tensor, u: torch.Tensor, v: torch.Tensor) -> torch.Tensor:
    """Link scores of an embedding table (fp32 [N, d], d a multiple of 32 up to 512) -> fp32 [P], out[i] = e_u[i] . e_v[i], one warp
    per pair with node2vec_step's dot routine: (u, v) and (v, u) give the same bits. One host read; raises IndexError for an id
    outside [0, N)."""
    _need_cuda(emb, u, v)
    assert emb.dim() == 2 and emb.dtype == torch.float32 and emb.is_contiguous(), "embedding_dot: emb must be contiguous fp32 [N, d]"
    d = _n2v_dim("embedding_dot", emb.shape[1])
    u, v = u.reshape(-1).to(torch.int64), v.reshape(-1).to(torch.int64)
    assert u.numel() == v.numel(), "embedding_dot: u / v size mismatch"
    n, P = emb.shape[0], u.numel()
    out = torch.empty(P, dtype=torch.float32, device=emb.device)
    if P == 0:
        return out
    nbad = int(((u < 0) | (u >= n) | (v < 0) | (v >= n)).sum())
    if nbad:
        raise IndexError(f"embedding_dot: {nbad} id(s) outside [0, {n})")
    (pu, su), (pv, sv) = _row(u), _row(v)
    check(lib.twowl_embedding_dot(emb.data_ptr(), n, d, pu, su, pv, sv, P, out.data_ptr(), _stream()), "embedding_dot")
    _count()
    return out


def node2vec(ptr: torch.Tensor, adj: torch.Tensor, dim: int = 128, walk_length: int = 80, walks_per_node: int = 10, window: int = 10,
             neg: int = 1, p: float = 1.0, q: float = 1.0, epochs: int = 1, batch_walks: int = 1024, lr: float = 0.01,
             seed: int = 0) -> Tuple[torch.Tensor, torch.Tensor]:
    """Train node2vec embeddings over a simple adjacency (simple_adjacency) -> (emb fp32 [N, dim], losses float64 [epochs], on the
    device). PyG Node2Vec's mini-batch recipe: emb starts N(0, 1); each epoch walks every node walks_per_node times in an order
    permuted by a generator seeded with `seed`, batch_walks walks at a time (node2vec_walks, index_base = the walk's index in the
    run), draws window * neg uniform negatives per token from the same generator (neg = negatives per positive pair) and runs one
    node2vec_step (lazy Adam, lr). losses[e] is the mean of epoch e's batch losses. The walk defaults are the node2vec paper's. No
    host read; two calls with the same arguments return the same bits on the same device. Raises ValueError for p, q as
    node2vec_walks does, dim as node2vec_step does, or a count < 1."""
    p, q = _n2v_pq("node2vec", p, q)
    dim = _n2v_dim("node2vec", dim)
    ints = dict(walk_length=walk_length, walks_per_node=walks_per_node, window=window, neg=neg, epochs=epochs, batch_walks=batch_walks)
    for k, val in ints.items():
        if int(val) < 1:
            raise ValueError(f"node2vec: {k} must be >= 1, got {val}")
    L, R, win, K, epochs, bw = (int(ints[k]) for k in ("walk_length", "walks_per_node", "window", "neg", "epochs", "batch_walks"))
    K *= win
    _need_cuda(ptr, adj)
    _check_graph("node2vec", ptr, adj)
    dev, n = ptr.device, ptr.numel() - 1
    gen = torch.Generator(device=dev)
    gen.manual_seed(int(seed))
    emb = torch.randn((n, dim), generator=gen, device=dev)
    exp_avg, exp_avg_sq = torch.zeros_like(emb), torch.zeros_like(emb)
    step = torch.zeros((), dtype=torch.int64, device=dev)
    losses = torch.zeros(epochs, dtype=torch.float64, device=dev)
    W = n * R
    if W == 0:
        return emb, losses
    nodes = torch.arange(n, device=dev).repeat(R)
    walk_seed = int(seed) & (2 ** 62 - 1)
    for e in range(epochs):
        starts = nodes[torch.randperm(W, generator=gen, device=dev)]
        total = torch.zeros((), dtype=torch.float64, device=dev)
        for b0 in range(0, W, bw):
            b1 = min(W, b0 + bw)
            walks = _n2v_walks(ptr, adj, starts[b0:b1], L, p, q, walk_seed, e * W + b0)
            negs = torch.randint(0, n, (b1 - b0, L, K), generator=gen, device=dev, dtype=torch.int32)
            total += _n2v_step(emb, exp_avg, exp_avg_sq, step, walks, negs, win, lr, (0.9, 0.999), 1e-8)
        losses[e] = total / -(-W // bw)
    return emb, losses


# ------------------------------------------------------------------------------ SEAL: enclosing subgraphs and DGCNN pieces

SEAL_MAX_WORKSPACE = 1 << 32   # default extraction workspace: 20 B per graph node for each CTA that runs at once
_SEAL_MAX_BLOCKS = 4 * 148


class SealBatch:
    """A batch of enclosing subgraphs (seal_subgraphs): node_ptr int64 [Q+1], nodes int64 [n] (global ids, ascending within a
    subgraph), z int32 [n] (DRNL labels), edge_index int64 [2, m] (ids into the batch's nodes, both directions, sorted by
    (row, col), block-diagonal by subgraph) and batch int64 [n] (each node's subgraph)."""
    __slots__ = ("node_ptr", "nodes", "z", "edge_index", "batch")

    def __init__(self, node_ptr, nodes, z, edge_index, batch):
        self.node_ptr, self.nodes, self.z, self.edge_index, self.batch = node_ptr, nodes, z, edge_index, batch

    @property
    def num_graphs(self) -> int:
        return self.node_ptr.numel() - 1


def _seal_args(fn: str, ptr, adj, src, dst, hops, max_nodes_per_hop, seed, index_base, max_workspace):
    _need_cuda(ptr, adj, src, dst)
    assert ptr.dim() == 1 and ptr.dtype == torch.int64 and ptr.is_contiguous(), f"{fn}: ptr must be contiguous int64 [N+1]"
    assert adj.dim() == 1 and adj.dtype == torch.int32 and adj.is_contiguous(), f"{fn}: adj must be contiguous int32"
    hops, cap = int(hops), int(max_nodes_per_hop)
    if hops not in (1, 2, 3):
        raise ValueError(f"{fn}: hops must be 1, 2 or 3, got {hops}")
    if not 0 <= cap < 2 ** 31:
        raise ValueError(f"{fn}: max_nodes_per_hop must be in [0, 2^31), got {cap}")
    if not 0 <= int(index_base) < 2 ** 31:
        raise ValueError(f"{fn}: index_base must be in [0, 2^31), got {index_base}")
    src, dst = src.reshape(-1).to(torch.int64), dst.reshape(-1).to(torch.int64)
    assert src.numel() == dst.numel(), f"{fn}: src / dst size mismatch"
    n, Q = ptr.numel() - 1, src.numel()
    budget = SEAL_MAX_WORKSPACE if max_workspace is None else int(max_workspace)
    per_block = lib.twowl_seal_workspace_bytes(n, 0, 2) - lib.twowl_seal_workspace_bytes(n, 0, 1)
    blocks = int(max(1, min(_SEAL_MAX_BLOCKS, max(Q, 1), budget // max(per_block, 1))))
    nb = lib.twowl_seal_workspace_bytes(n, Q, blocks)
    (ps, ss), (pd, sd) = (_row(src), _row(dst)) if Q else ((0, 1), (0, 1))
    return (ptr.data_ptr(), adj.data_ptr(), n, ps, ss, pd, sd, Q, int(index_base), hops, cap, int(seed) & (2 ** 64 - 1), blocks), \
        _ws(nb, ptr.device), nb, src, dst


def _seal_count(fn, args, ws, nb, dev):
    Q = args[7]
    node_ptr = torch.empty(Q + 1, dtype=torch.int64, device=dev)
    edge_ptr = torch.empty(Q + 1, dtype=torch.int64, device=dev)
    info = torch.empty(2, dtype=torch.int64, device=dev)
    check(lib.twowl_seal_count(*args, node_ptr.data_ptr(), edge_ptr.data_ptr(), info.data_ptr(), ws.data_ptr(), nb, _stream()), "seal_count")
    _count(1 + 2 * 3 + int(Q > 0))
    nbad, nself, n_nodes, n_edges = torch.cat((info, node_ptr[Q:], edge_ptr[Q:])).tolist()
    if nbad:
        raise IndexError(f"{fn}: {nbad} query id(s) outside [0, {args[2]})")
    if nself:
        raise ValueError(f"{fn}: {nself} query pair(s) with u == v")
    return node_ptr, edge_ptr, n_nodes, n_edges


def seal_subgraph_sizes(ptr: torch.Tensor, adj: torch.Tensor, src: torch.Tensor, dst: torch.Tensor, hops: int = 1,
                        max_nodes_per_hop: int = 0, seed: int = 0, index_base: int = 0,
                        max_workspace: Optional[int] = None) -> torch.Tensor:
    """The node count of each pair's enclosing subgraph (the count pass of seal_subgraphs alone) -> int64 [Q]."""
    args, ws, nb, src, dst = _seal_args("seal_subgraph_sizes", ptr, adj, src, dst, hops, max_nodes_per_hop, seed, index_base,
                                        max_workspace)
    node_ptr = _seal_count("seal_subgraph_sizes", args, ws, nb, ptr.device)[0]
    return node_ptr[1:] - node_ptr[:-1]


def seal_subgraphs(ptr: torch.Tensor, adj: torch.Tensor, src: torch.Tensor, dst: torch.Tensor, hops: int = 1,
                   max_nodes_per_hop: int = 0, seed: int = 0, index_base: int = 0,
                   max_workspace: Optional[int] = None) -> SealBatch:
    """SEAL's enclosing subgraph of each pair (src[q], dst[q]) over a simple adjacency (simple_adjacency) -> SealBatch.

    Nodes: {u, v}, then `hops` layers of unseen neighbours; a layer of more than max_nodes_per_hop nodes (0 = no cap) keeps the
    ones with the smallest hash of (seed, index_base + q, node), ties by id, and the dropped ones stay seen (the SEAL authors'
    k_hop_subgraph). The local order is ascending global id (PyG's relabel_nodes). Edges: the induced subgraph minus (u, v) and
    (v, u). z: DRNL labels (PyG's drnl_node_labeling, in integers). A caller that cuts one query list into several calls passes
    each call's offset as index_base to get the same subgraphs as one call. The result is bitwise repeatable and does not depend
    on max_workspace (default SEAL_MAX_WORKSPACE), which only bounds how many queries run at once. One host read (the counts);
    raises IndexError for an id outside [0, N) and ValueError for u == v, hops outside {1, 2, 3} or a negative cap."""
    fn = "seal_subgraphs"
    args, ws, nb, src, dst = _seal_args(fn, ptr, adj, src, dst, hops, max_nodes_per_hop, seed, index_base, max_workspace)
    dev = ptr.device
    node_ptr, edge_ptr, n_nodes, n_edges = _seal_count(fn, args, ws, nb, dev)
    nodes = torch.empty(n_nodes, dtype=torch.int64, device=dev)
    z = torch.empty(n_nodes, dtype=torch.int32, device=dev)
    edge_index = torch.empty((2, n_edges), dtype=torch.int64, device=dev)
    check(lib.twowl_seal_fill(*args, node_ptr.data_ptr(), edge_ptr.data_ptr(), n_edges, _p(nodes) if n_nodes else None,
                              _p(z) if n_nodes else None, _p(edge_index) if n_edges else None, ws.data_ptr(), nb, _stream()),
          "seal_fill")
    _count(2)
    Q = args[7]
    batch = torch.repeat_interleave(torch.arange(Q, device=dev), node_ptr[1:] - node_ptr[:-1], output_size=n_nodes)
    return SealBatch(node_ptr, nodes, z, edge_index, batch)


def label_gather(W: torch.Tensor, z: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out[m] (+)= W[:, z[m]] for W [C, L] (the linear map of one_hot(z, L) by W, without the one-hot matrix). With `out` the
    columns are added to it in place."""
    _need_cuda(W, z)
    W = W.contiguous()
    z = z.reshape(-1).to(torch.int64).contiguous()
    C, L = W.shape
    acc = out is not None
    if out is None:
        out = torch.empty((z.numel(), C), dtype=torch.float32, device=W.device)
    check(lib.twowl_label_gather(W.data_ptr(), C, L, z.data_ptr(), z.numel(), int(acc), out.data_ptr(), _stream()), "label_gather")
    _count()
    return out


def tanh_slice_fwd(h: torch.Tensor, out: torch.Tensor, off: int) -> torch.Tensor:
    """out[:, off:off + C] = tanh(h) for h [M, C] (out [M, ld] contiguous)."""
    _need_cuda(h, out)
    M, C = h.shape
    check(lib.twowl_tanh_slice_fwd(h.contiguous().data_ptr(), M, C, out.data_ptr(), out.shape[1], int(off), _stream()), "tanh_slice_fwd")
    _count()
    return out


def tanh_slice_bwd(g: torch.Tensor, y: torch.Tensor, off: int, C: int) -> torch.Tensor:
    """dh [M, C] = g[:, off:off + C] * (1 - y[:, off:off + C]^2) (g, y [M, ld] contiguous, of one shape)."""
    _need_cuda(g, y)
    assert g.shape == y.shape
    M = g.shape[0]
    dh = torch.empty((M, int(C)), dtype=torch.float32, device=g.device)
    check(lib.twowl_tanh_slice_bwd(g.contiguous().data_ptr(), y.data_ptr(), g.shape[1], int(off), M, int(C), dh.data_ptr(), _stream()),
          "tanh_slice_bwd")
    _count()
    return dh


def sortpool_fwd(X: torch.Tensor, gptr: torch.Tensor, k: int, key_col: int):
    """SortPooling: per graph the rows of X [n, D] by X[:, key_col] descending, ties by row, the first k -> (out [B, k, D] zero
    padded, idx int32 [B, k] = the rows taken, -1 for padding)."""
    _need_cuda(X, gptr)
    X = X.contiguous()
    B, D = gptr.numel() - 1, X.shape[1]
    out = torch.empty((B, int(k), D), dtype=torch.float32, device=X.device)
    idx = torch.empty((B, int(k)), dtype=torch.int32, device=X.device)
    check(lib.twowl_sortpool_fwd(X.data_ptr(), D, int(key_col), gptr.data_ptr(), B, int(k), out.data_ptr(), idx.data_ptr(), _stream()),
          "sortpool_fwd")
    _count()
    return out, idx


def sortpool_bwd(g: torch.Tensor, idx: torch.Tensor, n_rows: int) -> torch.Tensor:
    _need_cuda(g, idx)
    B, k, D = g.shape
    dX = torch.empty((int(n_rows), D), dtype=torch.float32, device=g.device)
    check(lib.twowl_sortpool_bwd(g.contiguous().data_ptr(), idx.data_ptr(), B, k, D, int(n_rows), dX.data_ptr(), _stream()), "sortpool_bwd")
    _count(2)
    return dX


def bias_act_fwd(Y: torch.Tensor, bias: torch.Tensor, B: int, pool: int, relu: bool, p_drop: float = 0.0, seed: int = 0) -> torch.Tensor:
    """Y [B * Lin, C] -> [B * (Lin // pool), C]: dropout_p(max over `pool` consecutive rows of act(Y + bias)), act = ReLU when relu,
    ties to the first row (nn.MaxPool1d(2, 2) after ReLU on Conv1d's [B, C, Lin] output, read transposed)."""
    _need_cuda(Y, bias)
    Y = Y.contiguous()
    C = Y.shape[1]
    Lin = Y.shape[0] // max(int(B), 1)
    out = torch.empty((int(B) * (Lin // int(pool)), C), dtype=torch.float32, device=Y.device)
    check(lib.twowl_bias_act_fwd(Y.data_ptr(), bias.contiguous().data_ptr(), int(B), max(Lin, 1), C, int(pool), int(relu), float(p_drop),
                                 int(seed), out.data_ptr(), _stream()), "bias_act_fwd")
    _count()
    return out


def bias_act_bwd(g: torch.Tensor, Y: torch.Tensor, bias: torch.Tensor, B: int, pool: int, relu: bool, p_drop: float = 0.0,
                 seed: int = 0) -> torch.Tensor:
    _need_cuda(g, Y, bias)
    C = Y.shape[1]
    Lin = Y.shape[0] // max(int(B), 1)
    dY = torch.empty_like(Y)
    check(lib.twowl_bias_act_bwd(g.contiguous().data_ptr(), Y.data_ptr(), bias.contiguous().data_ptr(), int(B), max(Lin, 1), C, int(pool),
                                 int(relu), float(p_drop), int(seed), dY.data_ptr(), _stream()), "bias_act_bwd")
    _count()
    return dY


def im2col_fwd(P: torch.Tensor, B: int, kw: int) -> torch.Tensor:
    """P [B * L1, C] (row b L1 + t = position t of sample b) -> [B * L2, C * kw], L2 = L1 - kw + 1, column c kw + j = P[b, p + j, c]."""
    _need_cuda(P)
    P = P.contiguous()
    C = P.shape[1]
    L1 = P.shape[0] // int(B)
    out = torch.empty((int(B) * (L1 - int(kw) + 1), C * int(kw)), dtype=torch.float32, device=P.device)
    check(lib.twowl_im2col_fwd(P.data_ptr(), int(B), L1, C, int(kw), out.data_ptr(), _stream()), "im2col_fwd")
    _count()
    return out


def im2col_bwd(g: torch.Tensor, B: int, L1: int, C: int, kw: int) -> torch.Tensor:
    _need_cuda(g)
    dP = torch.empty((int(B) * int(L1), int(C)), dtype=torch.float32, device=g.device)
    check(lib.twowl_im2col_bwd(g.contiguous().data_ptr(), int(B), int(L1), int(C), int(kw), dP.data_ptr(), _stream()), "im2col_bwd")
    _count()
    return dP
