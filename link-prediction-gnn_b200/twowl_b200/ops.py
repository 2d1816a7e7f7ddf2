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


def gcn_dinv_entries(ptr, col, M: int, entry_mask) -> torch.Tensor:
    """gcn_norm degree of a cached CSR minus the entries a per-entry mask removes."""
    _need_cuda(ptr, col, entry_mask)
    dinv = torch.empty(M, dtype=torch.float32, device=ptr.device)
    check(lib.twowl_gcn_dinv_entries(ptr.data_ptr(), col.data_ptr(), M, entry_mask.data_ptr(), dinv.data_ptr(), _stream()),
          "gcn_dinv_entries")
    _count()
    return dinv


def gather_u8(mask: torch.Tensor, ids: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """out[k] = mask[ids[k]] (uint8): a per-edge mask in the entry order of a CSR."""
    _need_cuda(mask, ids)
    if out is None:
        out = torch.empty(ids.numel(), dtype=torch.uint8, device=mask.device)
    assert out.dtype == torch.uint8 and out.is_contiguous() and out.numel() == ids.numel() and ids.is_contiguous()
    check(lib.twowl_gather_u8(mask.data_ptr(), ids.data_ptr(), ids.numel(), out.data_ptr(), _stream()), "gather_u8")
    _count()
    return out


def gcn_dinv_entries_rows(ptr, col, M: int, entry_mask, lo: int, hi: int, dinv: torch.Tensor) -> torch.Tensor:
    """gcn_dinv_entries for the node rows [lo, hi) only, written into dinv[lo:hi] (dinv: fp32, at least M elements)."""
    _need_cuda(ptr, col, entry_mask, dinv)
    assert dinv.dtype == torch.float32 and dinv.is_contiguous() and dinv.numel() >= M
    check(lib.twowl_gcn_dinv_entries_rows(ptr.data_ptr(), col.data_ptr(), M, entry_mask.data_ptr(), int(lo), int(hi), dinv.data_ptr(),
                                          _stream()), "gcn_dinv_entries_rows")
    _count()
    return dinv


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
    nbytes = col.numel() * (4 * C * (1 + int(pair_sum) + int(X2 is not None) + int(dual)) + 8 + 4 * int(dual)) + \
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


def pair_init_fwd(X, src32, dst32) -> torch.Tensor:
    _need_cuda(X, src32, dst32)
    R = src32.numel()
    out = torch.empty((R, X.shape[1]), dtype=torch.float32, device=X.device)
    with _P("pair_init_fwd", R * (12 * X.shape[1] + 8)):
        check(lib.twowl_pair_init_fwd(X.data_ptr(), src32.data_ptr(), dst32.data_ptr(), R, X.shape[1], out.data_ptr(),
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


def gn2_readout_bwd_prepare(xf, xr, sf, sr, pf, pr, p_drop: float, seed_f: int, seed_r: int, relu: bool, idx, w, dpred):
    """The row-sparse part of gn2_readout_bwd for a consumer that makes dxf / dxr on the fly (pair_dw_gn):
    -> (G [2L,C], head int32[M], next int32[2L], consts [8C], dparams_f, dparams_r [4C], dw [1,C], db [1])."""
    M, C = xf.shape
    dev = xf.device
    idx = idx.reshape(-1)
    L = idx.numel() // 2
    G = torch.empty((max(2 * L, 1), C), dtype=torch.float32, device=dev)
    head = torch.empty(M, dtype=torch.int32, device=dev)
    nxt = torch.empty(max(2 * L, 1), dtype=torch.int32, device=dev)
    consts = torch.empty(8 * C, dtype=torch.float32, device=dev)
    dpf = torch.empty(4 * C, dtype=torch.float32, device=dev)
    dpr = torch.empty(4 * C, dtype=torch.float32, device=dev)
    dw = torch.empty((1, C), dtype=torch.float32, device=dev)
    db = torch.empty(1, dtype=torch.float32, device=dev)
    nb = lib.twowl_gn2_readout_bwd_prepare_workspace_bytes(M, L, C)
    ws = _ws(nb, dev)
    p, s = _row(idx)
    dpred = dpred.contiguous()
    with _P("gn2_readout_bwd_prepare", M * 4 + L * (48 * C + 40)):
        check(lib.twowl_gn2_readout_bwd_prepare(xf.data_ptr(), xr.data_ptr(), M, C, sf.data_ptr(), sr.data_ptr(), pf[0].data_ptr(),
                                                pf[1].data_ptr(), pf[2].data_ptr(), pr[0].data_ptr(), pr[1].data_ptr(),
                                                pr[2].data_ptr(), float(p_drop), int(seed_f), int(seed_r), int(relu), p, s, L,
                                                w.data_ptr(), dpred.data_ptr(), G.data_ptr(), head.data_ptr(), nxt.data_ptr(),
                                                consts.data_ptr(), dpf.data_ptr(), dpr.data_ptr(), dw.data_ptr(), db.data_ptr(),
                                                ws.data_ptr(), nb, _stream()), "gn2_readout_bwd_prepare")
    _count(9)
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


def gn2_readout_bwd_rows(xf, xr, sf, sr, pf, pr, p_drop: float, seed_f: int, seed_r: int, relu: bool, idx, w, dpred):
    """Row part of gn2_readout_bwd_prepare over this rank's rows / positions:
    -> (G [2L,C], head int32[M], next int32[2L], colsums float64[6,C]) - colsums are summed over the ranks by the caller."""
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
    return G, head, nxt, colsums


def gn2_readout_bwd_finish(colsums, M_total: int, sf, sr, pf, pr):
    """-> (consts [8C], dparams_f, dparams_r [4C], dw [1,C], db [1]) from the rank-summed colsums of gn2_readout_bwd_rows."""
    C = colsums.shape[1]
    dev = colsums.device
    consts = torch.empty(8 * C, dtype=torch.float32, device=dev)
    dpf = torch.empty(4 * C, dtype=torch.float32, device=dev)
    dpr = torch.empty(4 * C, dtype=torch.float32, device=dev)
    dw = torch.empty((1, C), dtype=torch.float32, device=dev)
    db = torch.empty(1, dtype=torch.float32, device=dev)
    nb = lib.twowl_gn2_readout_bwd_finish_workspace_bytes(C)
    ws = _ws(nb, dev)
    check(lib.twowl_gn2_readout_bwd_finish(colsums.data_ptr(), int(M_total), C, sf.data_ptr(), sr.data_ptr(), pf[0].data_ptr(),
                                           pf[1].data_ptr(), pf[2].data_ptr(), pr[0].data_ptr(), pr[1].data_ptr(), pr[2].data_ptr(),
                                           consts.data_ptr(), dpf.data_ptr(), dpr.data_ptr(), dw.data_ptr(), db.data_ptr(),
                                           ws.data_ptr(), nb, _stream()), "gn2_readout_bwd_finish")
    _count(6)
    return consts, dpf, dpr, dw, db


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

def wedge_prepare(src32, dst_e32, E: int, R: int, N: int, blocked, in_ptr):
    dev = src32.device
    cnt = torch.empty(max(N, 1), dtype=torch.int32, device=dev)
    centre = torch.empty((2, R), dtype=torch.int32, device=dev)
    dinv = torch.empty((2, R), dtype=torch.float32, device=dev)
    selfw = torch.empty((2, R), dtype=torch.float32, device=dev)
    bnode = torch.empty((2, R), dtype=torch.int32, device=dev)
    check(lib.twowl_wedge_prepare(src32.data_ptr(), dst_e32.data_ptr(), E, R, N, _p(blocked), in_ptr.data_ptr(),
                                  cnt.data_ptr(), centre.data_ptr(), dinv.data_ptr(), selfw.data_ptr(), bnode.data_ptr(),
                                  _stream()), "wedge_prepare")
    _count(3)
    return cnt, centre, dinv, selfw, bnode


def wedge_prepare_rows(src32, dst_e32, E: int, R: int, N: int, blocked, in_ptr, lo: int, hi: int):
    """wedge_prepare for the pair rows [lo, hi) only -> (cnt [N], centre, dinv, selfw, bnode [2, hi - lo])."""
    dev = src32.device
    Rl = hi - lo
    cnt = torch.empty(max(N, 1), dtype=torch.int32, device=dev)
    centre = torch.empty((2, Rl), dtype=torch.int32, device=dev)
    dinv = torch.empty((2, Rl), dtype=torch.float32, device=dev)
    selfw = torch.empty((2, Rl), dtype=torch.float32, device=dev)
    bnode = torch.empty((2, Rl), dtype=torch.int32, device=dev)
    check(lib.twowl_wedge_prepare_rows(src32.data_ptr(), dst_e32.data_ptr(), E, R, N, _p(blocked), in_ptr.data_ptr(), int(lo), int(hi),
                                       cnt.data_ptr(), centre.data_ptr(), dinv.data_ptr(), selfw.data_ptr(), bnode.data_ptr(),
                                       _stream()), "wedge_prepare_rows")
    _count(3)
    return cnt, centre, dinv, selfw, bnode


def wedge_prepare_ranges(src32, dst_e32, E: int, R: int, N: int, blocked, in_ptr, r0, r1):
    """wedge_prepare for the pair rows r0 = [lo0, hi0) followed by r1 = [lo1, hi1) -> (cnt [N], centre, dinv, selfw, bnode
    [2, (hi0 - lo0) + (hi1 - lo1)]): one rank's block of the row-sharded step."""
    dev = src32.device
    Rl = (r0[1] - r0[0]) + (r1[1] - r1[0])
    cnt = torch.empty(max(N, 1), dtype=torch.int32, device=dev)
    centre = torch.empty((2, Rl), dtype=torch.int32, device=dev)
    dinv = torch.empty((2, Rl), dtype=torch.float32, device=dev)
    selfw = torch.empty((2, Rl), dtype=torch.float32, device=dev)
    bnode = torch.empty((2, Rl), dtype=torch.int32, device=dev)
    check(lib.twowl_wedge_prepare_ranges(src32.data_ptr(), dst_e32.data_ptr(), E, R, N, _p(blocked), in_ptr.data_ptr(), int(r0[0]),
                                         int(r0[1]), int(r1[0]), int(r1[1]), cnt.data_ptr(), centre.data_ptr(), dinv.data_ptr(),
                                         selfw.data_ptr(), bnode.data_ptr(), _stream()), "wedge_prepare_ranges")
    _count(4)
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
              want_moments: bool = False, out=None, pair_sum_out: bool = False):
    """out = sum_s (row_scale_s * A_s) B_s^T + sum_g coef_g * T_g[idx_g] + bias on tcgen05 (3xTF32).
    A, W, w_kn, row_scale: sequences of length nsrc; gathers: sequence of (T, idx int32, coef).
    Returns out, or (out, stats[2*Nd]) when stats_mean_scale is given (GraphNorm mean / inv_std of out), or
    (out, moments float64[2*Nd]) with want_moments (raw column sum / sum of squares, for a row-sharded caller).
    pair_sum_out: out is [M/2, Nd] and holds out[2k] + out[2k+1] (what the pair-init backward consumes: seg_reduce(x_pairs=True))."""
    nsrc = len(A)
    M, Kd = A[0].shape
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
                 pair_sum_out=int(pair_sum_out))
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
    nbytes = M * (4 * Kd * nsrc + 8 * len(gathers) + (4 * Nd + 8) * len(gathers)) + Mo * 4 * Nd
    with _P("pair_conv", nbytes):
        check(lib.twowl_pair_conv(ctypes.byref(a), _p(ws), nb, _stream()), "pair_conv")
    _count(1 if stats is None else 2)
    if moments is not None:
        return out, moments
    return out if stats is None else (out, stats)


# both directions of a pair layer in one pass over H (twowl_conv_args.dual). Off by default: bit-identical to the two launches
# and 20 GB less traffic at R-MAT scale, but at 128 output columns every epilogue warp serves two column blocks per tile and the
# second block's gather latency is exposed: 19.3 ms against 2 x 8.2 ms measured (DESIGN 4)
PAIR_CONV_DUAL = os.environ.get("TWOWL_PAIR_CONV_DUAL", "0") != "0"


def pair_conv_dual_supported(Kd: int, C: int) -> bool:
    return C % 32 == 0 and bool(lib.twowl_pair_conv_supported(Kd, 2 * C, 1))


def pair_conv_dual(A, Wf, Wr, rs_f, rs_r, gather_f, gather_r, bias_f, bias_r, ms_f, ms_r, eps: float = 1e-5, want_moments: bool = False):
    """Both directions of one pair layer (model.py:77) in ONE pass over A: O_d = rs_d * (A W_d^T) + coef_d * T_d[idx_d] + bias_d
    and the GraphNorm statistics of both. gather_d = (T_d [rows, C], idx_d int32 [M], coef_d [M]).
    -> (O_f, O_r, stats_f [2C], stats_r [2C]) or, with want_moments, (O_f, O_r, moments_f, moments_r float64 [2C])."""
    M, Kd = A.shape
    C = Wf.shape[0]
    dev = A.device
    _need_cuda(A, Wf, Wr)
    A = A.contiguous()
    W = torch.cat((Wf, Wr)).contiguous()
    bias = torch.cat((bias_f, bias_r))
    ms = torch.cat((ms_f, ms_r))
    Of = torch.empty((M, C), dtype=torch.float32, device=dev)
    Or = torch.empty((M, C), dtype=torch.float32, device=dev)
    a = ConvArgs(nsrc=1, ngather=2, Kd=Kd, Nd=2 * C, M=M, bias=bias.data_ptr(), out=Of.data_ptr(), out2=Or.data_ptr(), dual=1,
                 eps=float(eps))
    a.A[0], a.W[0], a.w_kn[0] = A.data_ptr(), W.data_ptr(), 0
    a.row_scale[0], a.row_scale[1] = rs_f.data_ptr(), rs_r.data_ptr()
    for g, (T, idx, coef) in enumerate((gather_f, gather_r)):
        a.T[g], a.tidx[g], a.tcoef[g] = T.data_ptr(), idx.data_ptr(), coef.data_ptr()
    stats = torch.empty(4 * C, dtype=torch.float32, device=dev)
    nb = lib.twowl_pair_conv_workspace_bytes(M, 2 * C)
    ws = _ws(nb, dev)
    a.stats, a.mean_scale = stats.data_ptr(), ms.data_ptr()
    moments = None
    if want_moments:
        moments = torch.zeros(4 * C, dtype=torch.float64, device=dev)
        a.moments = moments.data_ptr()
    nbytes = M * (4 * Kd + 2 * (4 * C + 4 * C + 16))
    with _P("pair_conv", nbytes):
        check(lib.twowl_pair_conv(ctypes.byref(a), ws.data_ptr(), nb, _stream()), "pair_conv (dual)")
    _count(2)
    if moments is not None:   # [sum(2C) | sumsq(2C)] -> per direction [sum(C) | sumsq(C)]
        m = moments.view(2, 2, C)
        return Of, Or, m[:, 0].reshape(-1), m[:, 1].reshape(-1)
    st = stats.view(2, 2, C)      # [mean(2C) | inv_std(2C)] -> per direction [mean(C) | inv_std(C)]
    return Of, Or, st[:, 0].reshape(-1), st[:, 1].reshape(-1)


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
    -> (dOf, dOr [M,C], dWf, dWr [C,C]). One pass: reads Of, Or, H, writes dOf, dOr (over Of, Or with inplace=True)."""
    _need_cuda(Of, Or, H)
    M, C = H.shape
    dOf, dOr = (Of, Or) if inplace else (torch.empty_like(Of), torch.empty_like(Or))
    dWf = torch.empty((C, C), dtype=torch.float32, device=H.device)
    dWr = torch.empty((C, C), dtype=torch.float32, device=H.device)
    nb = lib.twowl_pair_dw_workspace_bytes(M, C)
    ws = _ws(nb, H.device)
    with _P("pair_dw_gn", 20 * M * C + 12 * M):
        check(lib.twowl_pair_dw_gn(Of.data_ptr(), Or.data_ptr(), consts.data_ptr(), G.data_ptr(), head.data_ptr(), nxt.data_ptr(),
                                   float(p_drop), int(seed_f), int(seed_r), int(relu), rsf.data_ptr(), rsr.data_ptr(), H.data_ptr(),
                                   M, C, dOf.data_ptr(), dOr.data_ptr(), dWf.data_ptr(), dWr.data_ptr(), ws.data_ptr(), nb,
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


def graphnorm_bwd2(xf, xr, dout, sf, sr, pf, pr, p_drop: float, seed_f: int, seed_r: int, relu: bool):
    M, C = xf.shape
    dxf, dxr = torch.empty_like(xf), torch.empty_like(xr)
    dpf = torch.empty(4 * C, dtype=torch.float32, device=xf.device)
    dpr = torch.empty(4 * C, dtype=torch.float32, device=xf.device)
    nb = lib.twowl_graphnorm_bwd2_workspace_bytes(M, C)
    ws = _ws(nb, xf.device)
    with _P("graphnorm_bwd2", M * C * 4 * 8):
        check(lib.twowl_graphnorm_bwd2(xf.data_ptr(), xr.data_ptr(), dout.data_ptr(), M, C, sf.data_ptr(), sr.data_ptr(),
                                       pf[0].data_ptr(), pf[1].data_ptr(), pf[2].data_ptr(), pr[0].data_ptr(), pr[1].data_ptr(),
                                       pr[2].data_ptr(), float(p_drop), int(seed_f), int(seed_r), int(relu), dxf.data_ptr(),
                                       dxr.data_ptr(), dpf.data_ptr(), dpr.data_ptr(), ws.data_ptr(), nb, _stream()),
              "graphnorm_bwd2")
    _count(4)
    return dxf, dxr, dpf, dpr


def graphnorm_bwd2_sharded(xf, xr, dout, sf, sr, pf, pr, p_drop: float, seed_f: int, seed_r: int, relu: bool, M_total: int, all_reduce):
    """graphnorm_bwd2 over this rank's rows of a row-sharded pair table: the fp64 column sums [4,C] are summed over the ranks by
    `all_reduce` (a callable applied in place) between the two halves. -> (dxf, dxr, dparams_f, dparams_r) as graphnorm_bwd2."""
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
    all_reduce(colsums)
    dxf, dxr = torch.empty_like(xf), torch.empty_like(xr)
    dpf = torch.empty(4 * C, dtype=torch.float32, device=dev)
    dpr = torch.empty(4 * C, dtype=torch.float32, device=dev)
    nb2 = lib.twowl_graphnorm_bwd2_apply_workspace_bytes(C)
    ws2 = _ws(nb2, dev)
    with _P("graphnorm_bwd2", M * C * 4 * 5):
        check(lib.twowl_graphnorm_bwd2_apply(xf.data_ptr(), xr.data_ptr(), dout.data_ptr(), M, C, *ptrs, colsums.data_ptr(),
                                             int(M_total), dxf.data_ptr(), dxr.data_ptr(), dpf.data_ptr(), dpr.data_ptr(),
                                             ws2.data_ptr(), nb2, _stream()), "graphnorm_bwd2_apply")
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
