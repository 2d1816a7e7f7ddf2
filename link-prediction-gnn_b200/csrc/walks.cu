// walks.cu - global (path-based) link-prediction heuristics: truncated Katz and personalized PageRank, as pair scores and as
// top-k recommendations over all N nodes.
//
// Both indices are a few rounds of sparse propagation from a batch of source nodes, one column of a row-major fp32 [N, ld]
// operand Y per source. The propagation itself is twowl_seg_reduce on the simple adjacency with src_scale from
// twowl_walk_scale; this file holds what runs around it:
//   twowl_walk_scale    the per-node scale: beta (Katz) or alpha / d(w) (PPR, 0 for an isolated node)
//   twowl_walk_restart  Y[src[j], j] += value for the columns of a batch
//   twowl_walk_gather   out[dst[i]] = Y[v[i], col[i] - c_begin] for the pairs whose column lies in the batch
//   twowl_walk_topk     per column: s and N(s) excluded, the k largest positive scores, ties by ascending id. A radix select
//                       (four 8-bit digit passes; every column's 256-bin histogram in shared memory while Y streams row-major),
//                       a compaction of the entries above the threshold plus the lowest-id entries equal to it in ascending
//                       node order, then two stable radix sorts of the at most n_cols * k survivors (score key, then column).
// Integer atomics only (histogram counts): every result is bitwise repeatable, and a column's result depends on nothing but
// that column.
#include "common.cuh"

namespace twowl {

constexpr int kWalkThreads = 256;
constexpr int kWalkWarps = kWalkThreads / 32;
constexpr int kWalkTile = 256;      // rows of Y per warp task in the top-k passes: one warp reads 32 columns of each row (128 B)
constexpr int kWalkUnroll = 8;      // rows in flight per lane
constexpr uint32_t kWalkExcluded = 0xffffffffu;

// descending order-preserving key: larger scores get smaller keys; a score that is not > 0 (0, -0, negative, NaN) is excluded
__device__ __forceinline__ uint32_t walk_key(float x) { return x > 0.f ? ~auc_key(x) : kWalkExcluded; }

__global__ void __launch_bounds__(kWalkThreads) k_walk_scale(const int64_t* __restrict__ ptr, int64_t n, int method, float damping,
                                                             float* __restrict__ scale) {
  for (int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; w < n; w += (int64_t)gridDim.x * blockDim.x) {
    const int64_t d = ptr[w + 1] - ptr[w];
    scale[w] = method == TWOWL_WALK_KATZ ? damping : (d > 0 ? __fdiv_rn(damping, (float)d) : 0.f);
  }
}

__global__ void __launch_bounds__(kWalkThreads) k_walk_restart(float* __restrict__ Y, int64_t ld, int64_t n, const int64_t* __restrict__ src,
                                                               int64_t s_src, int64_t n_cols, float value) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_cols) return;
  const int64_t s = src[j * s_src];
  if (s >= 0 && s < n) Y[s * ld + j] += value;     // one thread per column: two columns sharing a source touch different words
}

// the pairs are ordered by column; each thread finds the batch's range [lo, hi) by binary search, then strides over it
__device__ __forceinline__ int64_t lower_bound_i64(const int64_t* a, int64_t n, int64_t x) {
  int64_t lo = 0, hi = n;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (__ldg(a + mid) < x) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}

__global__ void __launch_bounds__(kWalkThreads) k_walk_gather(const float* __restrict__ Y, int64_t ld, int64_t n, const int64_t* __restrict__ col,
                                                              const int64_t* __restrict__ v, const int64_t* __restrict__ dst, int64_t P,
                                                              int64_t c_begin, int64_t c_end, float* __restrict__ out) {
  const int64_t lo = lower_bound_i64(col, P, c_begin), hi = lower_bound_i64(col, P, c_end);
  for (int64_t i = lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t w = v[i];
    out[dst[i]] = (w >= 0 && w < n) ? Y[w * ld + (col[i] - c_begin)] : __int_as_float(0x7fffffff);
  }
}

// ---------------------------------------------------------------- top-k ---------------------------
// one warp per column: the source and its neighbours score 0, so that the selection below (score > 0) skips them
__global__ void __launch_bounds__(kWalkThreads) k_wt_exclude(const int64_t* __restrict__ ptr, const int32_t* __restrict__ adj, int64_t n,
                                                             float* __restrict__ Y, int64_t ld, const int64_t* __restrict__ src,
                                                             int64_t s_src, int64_t n_cols) {
  const int lane = threadIdx.x & 31;
  const int64_t j = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (j >= n_cols) return;
  const int64_t s = src[j * s_src];
  if (s < 0 || s >= n) return;
  if (lane == 0) Y[s * ld + j] = 0.f;
  for (int64_t e = ptr[s] + lane; e < ptr[s + 1]; e += 32) Y[(int64_t)__ldg(adj + e) * ld + j] = 0.f;
}

// the keys of rows [v0, v0 + kWalkTile) of column j (lane j % 32 of the warp), kWalkUnroll rows in flight; f(row, key)
template <typename F>
__device__ __forceinline__ void walk_tile_rows(const float* __restrict__ Y, int64_t ld, int64_t n, int64_t v0, int64_t j, F&& f) {
  const int64_t v1 = v0 + kWalkTile < n ? v0 + kWalkTile : n;
  for (int64_t v = v0; v < v1; v += kWalkUnroll) {
    float x[kWalkUnroll];
#pragma unroll
    for (int u = 0; u < kWalkUnroll; ++u) x[u] = (v + u < v1) ? __ldcs(Y + (v + u) * ld + j) : 0.f;
#pragma unroll
    for (int u = 0; u < kWalkUnroll; ++u)
      if (v + u < v1) f(v + u, walk_key(x[u]));
  }
}

// digit histogram of one radix pass: the entries whose higher digits equal the column's prefix. Shared layout [digit][lane]
// keeps the 32 lanes (= 32 columns) of a warp in 32 different banks.
__global__ void __launch_bounds__(kWalkThreads) k_wt_hist(const float* __restrict__ Y, int64_t ld, int64_t n, int64_t n_cols, int64_t ntiles,
                                                          int shift, const uint32_t* __restrict__ prefix, uint32_t* __restrict__ hist) {
  __shared__ uint32_t h[256 * 32];
  for (int i = threadIdx.x; i < 256 * 32; i += kWalkThreads) h[i] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t j = (int64_t)blockIdx.y * 32 + lane;
  if (j < n_cols) {
    const uint32_t hi_mask = shift == 24 ? 0u : ~0u << (shift + 8);
    const uint32_t pre = prefix[j] & hi_mask;
    for (int64_t t = (int64_t)blockIdx.x * kWalkWarps + warp; t < ntiles; t += (int64_t)gridDim.x * kWalkWarps)
      walk_tile_rows(Y, ld, n, t * kWalkTile, j, [&](int64_t, uint32_t key) {
        if ((key & hi_mask) == pre) atomicAdd(&h[((key >> shift) & 255u) * 32 + lane], 1u);
      });
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 256 * 32; i += kWalkThreads) {
    const int64_t jj = (int64_t)blockIdx.y * 32 + (i & 31);
    if (h[i] && jj < n_cols) atomicAdd(&hist[jj * 256 + (i >> 5)], h[i]);
  }
}

// one thread per column: the digit of the kk-th smallest key, and how many entries of that bucket are still to take
__global__ void __launch_bounds__(kWalkThreads) k_wt_select(const uint32_t* __restrict__ hist, int64_t n_cols, int shift, uint32_t kk,
                                                            uint32_t* __restrict__ prefix, uint32_t* __restrict__ krem) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n_cols) return;
  uint32_t want = shift == 24 ? kk : krem[j], pre = shift == 24 ? 0u : prefix[j], cum = 0;
  for (int b = 0; b < 256; ++b) {
    const uint32_t c = hist[j * 256 + b];
    if (cum + c >= want) {
      prefix[j] = pre | ((uint32_t)b << shift);
      krem[j] = want - cum;
      return;
    }
    cum += c;
  }
}

// per (column, tile): entries strictly below the threshold key, entries equal to it
__global__ void __launch_bounds__(kWalkThreads) k_wt_count(const float* __restrict__ Y, int64_t ld, int64_t n, int64_t n_cols, int64_t ntiles,
                                                           const uint32_t* __restrict__ thr, int64_t* __restrict__ lt, int64_t* __restrict__ eq) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t j = (int64_t)blockIdx.y * 32 + lane;
  if (j >= n_cols) return;
  const uint32_t T = thr[j];
  for (int64_t t = (int64_t)blockIdx.x * kWalkWarps + warp; t < ntiles; t += (int64_t)gridDim.x * kWalkWarps) {
    int64_t a = 0, b = 0;
    walk_tile_rows(Y, ld, n, t * kWalkTile, j, [&](int64_t, uint32_t key) {
      a += key < T;
      b += key == T;
    });
    lt[j * ntiles + t] = a;
    eq[j * ntiles + t] = b;
  }
}

// eq holds the flat exclusive scan of the equal counts: a tile takes the equal entries whose rank in the column is below krem
__device__ __forceinline__ int64_t wt_take(const int64_t* eq, int64_t ntiles, int64_t j, int64_t t, uint32_t krem, int64_t& budget) {
  budget = (int64_t)krem - (eq[j * ntiles + t] - eq[j * ntiles]);
  const int64_t c = eq[j * ntiles + t + 1] - eq[j * ntiles + t];
  return budget <= 0 ? 0 : (budget < c ? budget : c);
}

__global__ void __launch_bounds__(kWalkThreads) k_wt_take(int64_t n_cols, int64_t ntiles, const int64_t* __restrict__ eq,
                                                          const uint32_t* __restrict__ krem, int64_t* __restrict__ lt) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_cols * ntiles; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t j = i / ntiles;
    int64_t budget;
    lt[i] += wt_take(eq, ntiles, j, i - j * ntiles, krem[j], budget);
  }
}

// the survivors of each (column, tile) in ascending node order at the tile's offset (the flat scan of the per-tile totals:
// column j's kk survivors start at j * kk)
__global__ void __launch_bounds__(kWalkThreads) k_wt_write(const float* __restrict__ Y, int64_t ld, int64_t n, int64_t n_cols, int64_t ntiles,
                                                           const uint32_t* __restrict__ thr, const uint32_t* __restrict__ krem,
                                                           const int64_t* __restrict__ off, const int64_t* __restrict__ eq,
                                                           uint32_t* __restrict__ keys, uint32_t* __restrict__ pos, uint32_t* __restrict__ node) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t j = (int64_t)blockIdx.y * 32 + lane;
  if (j >= n_cols) return;
  const uint32_t T = thr[j];
  for (int64_t t = (int64_t)blockIdx.x * kWalkWarps + warp; t < ntiles; t += (int64_t)gridDim.x * kWalkWarps) {
    int64_t p = off[j * ntiles + t], budget;
    wt_take(eq, ntiles, j, t, krem[j], budget);
    walk_tile_rows(Y, ld, n, t * kWalkTile, j, [&](int64_t v, uint32_t key) {
      if (key < T || (key == T && budget-- > 0)) {
        keys[p] = key, pos[p] = (uint32_t)p, node[p] = (uint32_t)v;
        ++p;
      }
    });
  }
}

__global__ void __launch_bounds__(kWalkThreads) k_wt_colkeys(const uint32_t* __restrict__ pos, int64_t M, uint32_t kk, uint32_t* __restrict__ keys,
                                                             uint32_t* __restrict__ vals) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < M; i += (int64_t)gridDim.x * blockDim.x) {
    keys[i] = pos[i] / kk;
    vals[i] = pos[i];
  }
}

// row q_begin + j of (ids, scores): the column's survivors in (score descending, id ascending) order, then -1 / NaN
__global__ void __launch_bounds__(kWalkThreads) k_wt_out(const float* __restrict__ Y, int64_t ld, const uint32_t* __restrict__ order,
                                                         const uint32_t* __restrict__ node, int64_t n_cols, int64_t kk, int64_t k,
                                                         int64_t q_begin, int64_t* __restrict__ ids, float* __restrict__ scores) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_cols * k; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t j = i / k, r = i - j * k;
    int64_t id = -1;
    float x = __int_as_float(0x7fffffff);
    if (r < kk) {
      const int64_t v = node[order[j * kk + r]];
      const float y = Y[v * ld + j];
      if (y > 0.f) id = v, x = y;
    }
    ids[q_begin * k + i] = id;
    scores[q_begin * k + i] = x;
  }
}

struct WalkTopkWs {
  uint32_t *hist, *prefix, *krem;
  int64_t *lt, *eq;
  void* sws;
  uint32_t *k0, *v0, *k1, *v1, *node;
  void* rws;
};

static int64_t walk_tiles(int64_t n) { return cdiv(n > 0 ? n : 1, kWalkTile); }

// the workspace of twowl_walk_topk laid out from `base` (NULL: only its size is wanted)
static size_t walk_topk_carve(void* base, int64_t n, int64_t n_cols, int64_t k, WalkTopkWs& w) {
  const int64_t nc = n_cols > 0 ? n_cols : 1, kk = k < n ? k : n, M = nc * (kk > 0 ? kk : 1), F = nc * walk_tiles(n);
  Carver c(base);
  w.hist = c.take<uint32_t>(4 * 256 * nc);
  w.prefix = c.take<uint32_t>(nc);
  w.krem = c.take<uint32_t>(nc);
  w.lt = c.take<int64_t>(F + 1);
  w.eq = c.take<int64_t>(F + 1);
  w.sws = c.take<char>(scan_workspace_bytes(F));
  w.k0 = c.take<uint32_t>(M);
  w.v0 = c.take<uint32_t>(M);
  w.k1 = c.take<uint32_t>(M);
  w.v1 = c.take<uint32_t>(M);
  w.node = c.take<uint32_t>(M);
  w.rws = c.take<char>(radix_workspace_bytes(M));
  return c.off;
}

}  // namespace twowl

using namespace twowl;

extern "C" int twowl_walk_scale(const int64_t* ptr, int64_t num_nodes, int32_t method, float damping, float* scale, void* stream) {
  TW_CHECK_ARG(num_nodes >= 0 && num_nodes < 0x7fffffffLL, "walk_scale: bad sizes (0 <= num_nodes < 2^31 - 1)");
  TW_CHECK_ARG(method == TWOWL_WALK_KATZ || method == TWOWL_WALK_PPR, "walk_scale: method must be 0 (katz) or 1 (ppr)");
  TW_CHECK_ARG(method == TWOWL_WALK_KATZ ? (damping > 0.f && damping <= 3.4e38f) : (damping > 0.f && damping < 1.f),
               "walk_scale: damping must be finite and > 0 (katz) or in (0, 1) (ppr)");
  TW_CHECK_ARG(num_nodes == 0 || (ptr && scale), "walk_scale: null pointer");
  if (num_nodes == 0) return 0;
  k_walk_scale<<<grid_for(num_nodes, kWalkThreads), kWalkThreads, 0, (cudaStream_t)stream>>>(ptr, num_nodes, method, damping, scale);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" int twowl_walk_restart(float* Y, int64_t ld, int64_t num_nodes, const int64_t* src, int64_t s_src, int64_t n_cols, float value,
                                  void* stream) {
  TW_CHECK_ARG(num_nodes >= 0 && num_nodes < 0x7fffffffLL && n_cols >= 0 && ld >= n_cols, "walk_restart: bad sizes (0 <= n_cols <= ld)");
  TW_CHECK_ARG(n_cols == 0 || num_nodes == 0 || (Y && src), "walk_restart: null pointer");
  if (n_cols == 0 || num_nodes == 0) return 0;
  k_walk_restart<<<(int)cdiv(n_cols, kWalkThreads), kWalkThreads, 0, (cudaStream_t)stream>>>(Y, ld, num_nodes, src, s_src, n_cols, value);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" int twowl_walk_gather(const float* Y, int64_t ld, int64_t num_nodes, const int64_t* col, const int64_t* v, const int64_t* dst,
                                 int64_t P, int64_t c_begin, int64_t c_end, float* out, void* stream) {
  TW_CHECK_ARG(num_nodes >= 0 && num_nodes < 0x7fffffffLL && P >= 0 && 0 <= c_begin && c_begin <= c_end && c_end - c_begin <= ld,
               "walk_gather: bad sizes (0 <= P, 0 <= c_begin <= c_end <= c_begin + ld)");
  TW_CHECK_ARG(P == 0 || (Y && col && v && dst && out), "walk_gather: null pointer");
  if (P == 0 || c_begin == c_end) return 0;
  k_walk_gather<<<grid_for(P, kWalkThreads), kWalkThreads, 0, (cudaStream_t)stream>>>(Y, ld, num_nodes, col, v, dst, P, c_begin, c_end, out);
  TW_LAUNCH_CHECK();
  return 0;
}

extern "C" size_t twowl_walk_topk_workspace_bytes(int64_t num_nodes, int64_t n_cols, int64_t k) {
  WalkTopkWs w;
  return walk_topk_carve(nullptr, num_nodes > 0 ? num_nodes : 0, n_cols, k > 0 ? k : 1, w);
}

extern "C" int twowl_walk_topk(const int64_t* ptr, const int32_t* adj, int64_t num_nodes, float* Y, int64_t ld, const int64_t* src,
                               int64_t s_src, int64_t n_cols, int64_t k, int64_t Q, int64_t q_begin, int64_t* ids, float* scores, void* ws,
                               size_t ws_bytes, void* stream) {
  TW_CHECK_ARG(num_nodes >= 0 && num_nodes < 0x7fffffffLL && n_cols >= 0 && ld >= n_cols && 0 <= q_begin && q_begin + n_cols <= Q,
               "walk_topk: bad sizes (0 <= n_cols <= ld, 0 <= q_begin, q_begin + n_cols <= Q)");
  TW_CHECK_ARG(k >= 1 && k < 0x7fffffffLL && Q * k < (1LL << 60), "walk_topk: k must be in [1, 2^31) with Q * k < 2^60");
  const int64_t kk = k < num_nodes ? k : num_nodes;
  TW_CHECK_ARG(n_cols * kk < 0x80000000LL, "walk_topk: n_cols * min(k, num_nodes) must be < 2^31");
  TW_CHECK_ARG(n_cols == 0 || (ptr && ids && scores && src && (num_nodes == 0 || Y)), "walk_topk: null pointer");   // adj: NULL when nnz = 0
  TW_CHECK_WS(ws_bytes, twowl_walk_topk_workspace_bytes(num_nodes, n_cols, k));
  if (n_cols == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t n = num_nodes;
  WalkTopkWs w;
  walk_topk_carve(ws, n, n_cols, k, w);
  if (kk > 0) {
    const int64_t ntiles = walk_tiles(n), nslabs = cdiv(n_cols, 32), M = n_cols * kk;
    k_wt_exclude<<<(int)cdiv(n_cols * 32, kWalkThreads), kWalkThreads, 0, s>>>(ptr, adj, n, Y, ld, src, s_src, n_cols);
    TW_LAUNCH_CHECK();
    TW_CUDA(cudaMemsetAsync(w.hist, 0, (size_t)4 * 256 * n_cols * sizeof(uint32_t), s));
    const dim3 grid((unsigned)std::max<int64_t>(1, std::min(cdiv(ntiles, kWalkWarps), cdiv(4 * kNumSMs, nslabs))), (unsigned)nslabs);
    for (int pass = 0; pass < 4; ++pass) {
      const int shift = 24 - 8 * pass;
      uint32_t* h = w.hist + (size_t)pass * 256 * n_cols;
      k_wt_hist<<<grid, kWalkThreads, 0, s>>>(Y, ld, n, n_cols, ntiles, shift, w.prefix, h);
      k_wt_select<<<(int)cdiv(n_cols, kWalkThreads), kWalkThreads, 0, s>>>(h, n_cols, shift, (uint32_t)kk, w.prefix, w.krem);
      TW_LAUNCH_CHECK();
    }
    const int64_t F = n_cols * ntiles;
    k_wt_count<<<grid, kWalkThreads, 0, s>>>(Y, ld, n, n_cols, ntiles, w.prefix, w.lt, w.eq);
    TW_LAUNCH_CHECK();
    if (int rc = scan_exclusive_i64(w.eq, w.eq, F, w.sws, s)) return rc;
    k_wt_take<<<grid_for(F, kWalkThreads), kWalkThreads, 0, s>>>(n_cols, ntiles, w.eq, w.krem, w.lt);
    TW_LAUNCH_CHECK();
    if (int rc = scan_exclusive_i64(w.lt, w.lt, F, w.sws, s)) return rc;
    k_wt_write<<<grid, kWalkThreads, 0, s>>>(Y, ld, n, n_cols, ntiles, w.prefix, w.krem, w.lt, w.eq, w.k0, w.v0, w.node);
    TW_LAUNCH_CHECK();
    // stably by the score key, then stably by the column: each column's survivors by (score descending, node ascending)
    if (int rc = radix_sort_pairs(w.k0, w.v0, w.k1, w.v1, M, 32, w.rws, s)) return rc;
    k_wt_colkeys<<<grid_for(M, kWalkThreads), kWalkThreads, 0, s>>>(w.v1, M, (uint32_t)kk, w.k0, w.v0);
    TW_LAUNCH_CHECK();
    if (int rc = radix_sort_pairs(w.k0, w.v0, w.k1, w.v1, M, bits_for_value(n_cols - 1), w.rws, s)) return rc;
  }
  k_wt_out<<<grid_for(n_cols * k, kWalkThreads), kWalkThreads, 0, s>>>(Y, ld, w.v1, w.node, n_cols, kk, k, q_begin, ids, scores);
  TW_LAUNCH_CHECK();
  return 0;
}
